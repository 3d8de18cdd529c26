"""CPU tests of the C-ABI boundary: the library loads, exports every symbol include/whisper_b200.h
declares, its host-side logic (beam.rs / windowing restated in C++) matches the oracle, and
compute entry points fail loudly without a GPU (no CPU fallback)."""
import ctypes as C
import json
import re
from pathlib import Path

import numpy as np
import pytest
import torch

import wb200  # noqa: F401
from oracle import beam as o_beam, transcribe as o_tr
from whisper_burn_b200 import audio, beam, ffi, transcribe

ROOT = Path(__file__).resolve().parent.parent
G = Path(__file__).resolve().parent / "golden"


@pytest.fixture(scope="module", autouse=True)
def built():
    if not ffi.library_path().exists():
        import __graft_entry__ as ge
        ge.build()


def test_header_symbols_exported():
    header = (ROOT / "include" / "whisper_b200.h").read_text()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)      # drop comments
    declared = set(re.findall(r"\b(wb_[a-z0-9_]+)\s*\(", header))
    assert declared == set(ffi.SYMBOLS), declared ^ set(ffi.SYMBOLS)
    lib = ffi.lib()
    for name in declared:
        assert getattr(lib, name) is not None
    assert b"sm_100a" in lib.wb_version()


def test_max_waveform_samples_and_windows_match_oracle():
    for n in (0, 1, 10, 1490, 2990):
        assert audio.max_waveform_samples(n) == 160 * (n + 1) - 1
    for n_samples in (0, 1, 399, 238559, 238560, 480000, 1000000):
        assert transcribe.window_bounds(n_samples, 16000, 238559) == o_tr.window_bounds(n_samples, 16000, 238559)
    assert transcribe.window_bounds(5000, 16000, 100) == o_tr.window_bounds(5000, 16000, 100)   # shift saturates to 1


def test_get_top_elements_matches_beam_rs_table():
    for c in json.loads((G / "beam_ties.json").read_text()):
        assert beam.get_top_elements(c["scores"], c["num"]) == c["expect"]
    rng = np.random.default_rng(0)
    for _ in range(200):
        s = rng.integers(-4, 5, size=int(rng.integers(0, 40))).astype(np.float64)
        k = int(rng.integers(1, 7))
        assert beam.get_top_elements(s, k) == o_beam.get_top_elements(list(range(len(s))), lambda i: s[i], k)


def test_find_chunk_overlap_matches_oracle():
    rng = np.random.default_rng(1)
    for _ in range(300):
        a = [int(v) for v in rng.integers(0, 6, size=int(rng.integers(0, 60)))]
        b = [int(v) for v in rng.integers(0, 6, size=int(rng.integers(0, 60)))]
        assert transcribe.find_chunk_overlap(a, b, 40, 3) == o_tr.find_chunk_overlap(a, b, 40, 3)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU error path")
def test_compute_fails_loudly_without_gpu():
    with pytest.raises(ffi.WbError) as e:
        audio.prep_audio(np.zeros((1, 1600), np.float32))
    assert e.value.code == ffi.WB_ERR_CUDA and "no CPU fallback" in e.value.msg
    h = C.c_void_p()
    dims = ffi.Dims(80, 1500, 128, 2, 2, 1024, 448, 128, 2, 2)
    assert ffi.lib().wb_model_create(C.byref(dims), 0, C.byref(h)) == ffi.WB_ERR_CUDA


def test_contract_violations_are_invalid_arg():
    # the reference panics (audio.rs:292); the ABI reports WB_ERR_INVALID_ARG before touching the device
    with pytest.raises(ffi.WbError) as e:
        audio.prep_audio(np.zeros((1, 399), np.float32))
    assert e.value.code == ffi.WB_ERR_INVALID_ARG


def test_npy_tree_probe_reads_reference_format(tmp_path):
    """The reference's model-file format (python/dump.py:120-213 / src/model/load.rs:19-53): dims come from the tree."""
    from whisper_burn_b200 import npytree, synth
    dims, w_np = synth.make_weights("test-a", seed=1)
    npytree.save_npy_tree(tmp_path, dims, w_np)
    got = npytree.probe(tmp_path)
    assert got == dims
    raw = np.load(tmp_path / "encoder/conv1/weight.npy")
    assert raw.dtype == np.float32 and list(raw[:3]) == [dims.n_audio_state, 80, 3]      # [dims..., values...]
    assert list(np.load(tmp_path / "encoder/ln_post/eps.npy")) == [1.0, np.float32(1e-5)]   # scalars as [1.0, value]
    (tmp_path / "encoder/n_mels.npy").unlink()
    with pytest.raises(ffi.WbError) as e:
        npytree.probe(tmp_path)
    assert e.value.code == ffi.WB_ERR_STATE and "n_mels" in e.value.msg


@pytest.mark.parametrize("beam_size,quant", [(1, 0), (5, 0), (5, 3), (3, 2)])
def test_host_beam_search_matches_oracle(beam_size, quant):
    """The complete C++ host search (host/beam.hpp: step, finished-beam carry, earlier-wins / last-max tie-breaks, beam.rs:9-110)
    against the oracle's restatement, driven by the same table-defined `next`; quant > 0 rounds the log-probs to create exact ties."""
    from oracle import beam as o_beam
    from whisper_burn_b200 import beam as w_beam
    rng = np.random.default_rng(100 + beam_size * 7 + quant)
    n_ctx, V, eot = 37, 23, 22
    for trial in range(6):
        table = np.log(rng.dirichlet(np.ones(V) * 0.7, size=n_ctx))
        if quant:
            table = np.round(table, quant)
        table[:, eot] += 0.5 * trial                     # later trials finish early

        def next_fn(beams):
            return [[(v, b.log_prob + float(table[(b.seq[-1] * 131 + len(b.seq)) % n_ctx, v])) for v in range(V)] for b in beams]

        want = o_beam.beam_search([o_beam.BeamNode(seq=[3], log_prob=0.0)], next_fn, lambda s: s[-1] == eot, beam_size, 12)
        assert w_beam.beam_search_table(table, 3, eot, beam_size, 12) == want


def test_npy_tree_rejects_malformed_files(tmp_path):
    """load.rs:19-27 trusts the leading dims; the C++ reader checks them (size mismatch, dtype, magic) and says which file."""
    from whisper_burn_b200 import npytree, synth
    dims, w_np = synth.make_weights("test-a", seed=1)
    npytree.save_npy_tree(tmp_path, dims, w_np)
    p = tmp_path / "decoder/token_embedding/weight.npy"
    good = np.load(p)
    np.save(p, good[:-3])                                   # payload shorter than its leading dims
    with pytest.raises(ffi.WbError) as e:
        npytree.probe(tmp_path)
    assert e.value.code == ffi.WB_ERR_INVALID_ARG and "token_embedding" in e.value.msg
    np.save(p, good.astype(np.float64))                     # npy::NpyData<f32> (load.rs:19): f32 only
    with pytest.raises(ffi.WbError) as e:
        npytree.probe(tmp_path)
    assert "float32" in e.value.msg
    p.write_bytes(b"not an npy file")
    with pytest.raises(ffi.WbError) as e:
        npytree.probe(tmp_path)
    assert e.value.code == ffi.WB_ERR_INVALID_ARG


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU port of the reference path): ONE JSON line with the contract's keys, no GPU needed."""
    import json, subprocess, sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    r = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--max-depth", "3",
                        "--cpu-baseline-windows", "1"], capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["metric"] == "audio-seconds/sec" and j["unit"] == "audio-s/s" and j["higher_is_better"] is True
    assert j["value"] > 0 and j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1
    assert j["e2e"] == {"value": j["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_integration_excerpts_are_literal_and_shim_symbols_exist():
    """INTEGRATION.md quotes rust/src/lib.rs literally, and every wb_* symbol the Rust shim binds is declared in the header
    (and therefore exported: test_header_symbols_match_library)."""
    import re
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    lib = (root / "rust" / "src" / "lib.rs").read_text()
    md = (root / "INTEGRATION.md").read_text()
    blocks = re.findall(r"<!-- excerpt:\w+ -->\n```rust\n(.*?)```\n<!-- /excerpt -->", md, flags=re.S)
    assert len(blocks) == 2
    for b in blocks:
        assert b in lib, "INTEGRATION.md excerpt drifted from rust/src/lib.rs"
    header = (root / "include" / "whisper_b200.h").read_text()
    for sym in set(re.findall(r"pub fn (wb_\w+)\(", lib)):
        assert re.search(r"\b" + sym + r"\(", header), f"{sym} bound by the shim but not declared in the header"


def test_repetition_heuristics_match_oracle():
    """transcribe.rs:385-447 (compiled but unused by the reference's live path): C++ vs the oracle restatement on random
    low-entropy sequences, crafted periodic tails, empty / short inputs, and the inputs on which the reference panics."""
    import numpy as np
    import pytest
    from oracle import transcribe as o_tr
    from whisper_burn_b200 import transcribe
    rng = np.random.default_rng(5)
    seqs = [[], [7], [1, 2, 3], [5] * 12, [1, 2, 3, 1, 2, 3, 1, 2, 3, 1, 2, 3, 1, 2, 3], [9, 8, 1, 2, 1, 2, 1, 2, 1, 2, 1, 2],
            [4, 4, 1, 2, 3, 4, 5, 0, 1, 2, 3, 4, 5, 7, 1, 2, 3, 4, 5, 6, 6, 1, 2, 3, 4, 5, 1, 2, 3, 4, 5]]
    for _ in range(300):
        n = int(rng.integers(0, 40))
        base = rng.integers(0, 3, size=n).tolist()
        if n > 6 and rng.random() < 0.5:      # periodic tail
            p = int(rng.integers(1, 5))
            base = base[:n // 2] + (base[:p] * 12)[:n - n // 2]
        seqs.append(base)

    def both(fn_ours, fn_oracle, *a):
        try:
            want = fn_oracle(*a)
        except ValueError:
            with pytest.raises(ValueError):
                fn_ours(*a)
            return
        assert fn_ours(*a) == want, (a, want)

    for s in seqs:
        for period in range(0, 7):
            both(transcribe.first_repetition_end, o_tr.first_repetition_end, s, period)
        for reps in range(0, 5):
            both(transcribe.repetition_period, o_tr.repetition_period, s, reps)
        for win in range(0, 6):
            for cnt in range(0, 5):
                both(transcribe.find_repeated_tokens_index, o_tr.find_repeated_tokens_index, s, win, cnt)
    # the reference's own settings (transcribe.rs:359-360): window 5, four repeats
    s = [4, 4, 1, 2, 3, 4, 5, 0, 1, 2, 3, 4, 5, 7, 1, 2, 3, 4, 5, 6, 6, 1, 2, 3, 4, 5, 1, 2, 3, 4, 5]
    assert transcribe.find_repeated_tokens_index(s, 5, 4) == (2, 8)
    assert transcribe.repetition_period([0, 9] + [1, 2, 3] * 5, 4) == 3


def test_bench_algorithmic_bytes_tiny_en_headline():
    """The numerator of the bench line's roofline (SURVEY.md 8d) for the headline workload, evaluated by hand: tiny.en, the three
    reference windows of a 30 s chunk (750 + 750 + 314 encoder positions), fp16-exact weights, fp32 K/V, 103 positions."""
    import importlib.util
    from pathlib import Path
    from whisper_burn_b200 import synth
    spec = importlib.util.spec_from_file_location("bench_mod", Path(__file__).resolve().parent.parent / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    dims = synth.MODEL_DIMS["tiny.en"]
    lens = [238559, 238559, 480000 - 381118]
    d, L, V = 384, 4, 51864
    weights = L * 14 * d * d * 2                       # 16.5 MB of layer weights per position
    cross = L * 2 * (750 + 750 + 314) * d * 4          # 22.3 MB of cross K/V per position
    self_kv = sum(L * 2 * (t + 1) * d * 4 * 3 for t in range(103))
    want = (weights + cross) * 103 + 100 * V * d * 2 + self_kv
    assert bench.algorithmic_bytes(dims, lens, 2, 4, 100) == want == 8177565696
    # the fp16 cache halves the K/V terms only
    assert bench.algorithmic_bytes(dims, lens, 2, 2, 100) == weights * 103 + (cross * 103 + self_kv) // 2 + 100 * V * d * 2 == 6930886656


def test_bench_dump_outputs_format_and_steps_argument(tmp_path):
    """`bench.py --dump-outputs DIR` writes each token id list of lists as a float64 [n, longest] matrix padded with -1;
    `--steps` below 1 is refused rather than silently raised to 1."""
    import importlib.util
    import subprocess
    import sys
    spec = importlib.util.spec_from_file_location("bench_mod", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    bench.write_outputs(tmp_path / "out", {"0_tiny.en_1chunks_f32_window_tokens": [[50257, 50259, 7], [50257]], "empty": []})
    m = np.load(tmp_path / "out" / "0_tiny.en_1chunks_f32_window_tokens.npy")
    assert m.dtype == np.float64 and m.tolist() == [[50257, 50259, 7], [50257, -1, -1]]
    assert np.load(tmp_path / "out" / "empty.npy").shape == (0, 0)
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "0"], capture_output=True, text=True,
                       timeout=120, cwd=ROOT)
    assert r.returncode == 2 and "--steps" in r.stderr
