"""The C-ABI library loads and exports every symbol include/emb200.h declares (no GPU needed)."""
import ctypes as C
import os
import re

import pytest

from em_model_manned_bayes_b200 import _lib as L
from helpers import ROOT


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "emb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(emb_[A-Za-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = L.lib()
    names = declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(L.EXPORTED) == names
    assert lib.emb_abi_version() == 2


def test_struct_layouts_match_header_sizes():
    # sizes computed from the header's field list (natural alignment)
    assert C.sizeof(L.Rng) == 16
    assert C.sizeof(L.TrackOut) == 7 * 8
    assert C.sizeof(L.SampleOpts) == 24 * 4 + 4 * 4 + 2 * 24 * 8 + 4 + 4 + 8 * 2 * 8 + 4 * 3 + 4 + 8 + 8 + 8
    assert C.sizeof(L.ModelInfo) % 8 == 0


def test_rng_word_matches_oracle_stream():
    from oracle import philox as px
    lib = L.lib()
    for (seed, sample, attempt, purpose, index, sub, lane) in [(1, 0, 0, 1, 0, 0, 0), (2 ** 63 + 5, 12345678901, 3, 2, 77, 0, 3),
                                                             (42, 2 ** 40, 65535, 3, 599, 1, 2)]:
        got = lib.emb_rng_word(seed, sample, attempt, purpose, index, sub, lane)
        want = int(px.word(seed, sample, attempt, purpose, index, lane, sub=sub))
        assert got == want


def test_no_cpu_fallback_without_gpu(model_paths):
    """Sampling must fail loudly (EMB_E_CUDA) when no device is present -- never silently compute on the CPU."""
    lib = L.lib()
    if lib.emb_device_count() > 0:
        pytest.skip("a CUDA device is present")
    from em_model_manned_bayes_b200.model import EncounterModel
    m = EncounterModel(model_paths["balloon_v1"])
    with pytest.raises(L.EmbError) as ei:
        m.sample_initial(4, seed=1)
    assert ei.value.code == L.EMB_E_CUDA


def test_mex_gateway_source_matches_the_header():
    """matlab/emb_mex.cpp cannot be built here (no MATLAB), but it must at least compile against include/emb200.h:
    syntax- and type-check it with a declarations-only stand-in for mex.h (tests/stubs/mex.h)."""
    import subprocess
    r = subprocess.run(["g++", "-std=c++17", "-fsyntax-only", "-Wall", "-I", os.path.join(ROOT, "tests", "stubs"),
                        "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "matlab", "emb_mex.cpp")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    src = open(os.path.join(ROOT, "matlab", "emb_mex.cpp")).read()
    for fn in ("emb_model_load", "emb_model_from_arrays", "emb_sample_track_events_packed", "emb_sample_tracks_multi", "emb_set_prior", "emb_sample_initial", "emb_sample_tracks", "emb_sample_track_events",
               "emb_terminal_propagate", "emb_terminal_screen", "emb_tracks_integrate"):
        assert fn + "(" in src, fn


def test_terminal_structs_match_header_sizes():
    assert C.sizeof(L.DynLimits) == 5 * 8
    assert C.sizeof(L.TerminalModels) == 10 * 8
    assert C.sizeof(L.TrajOut) == 2 * 8


MATLAB_DIR = os.path.join(ROOT, "matlab")


def _upstream():
    """What these tests need of the upstream classes and functions (tests/golden/upstream_reference.json)."""
    import json
    return json.load(open(os.path.join(ROOT, "tests", "golden", "upstream_reference.json")))


def _glue_sources():
    for f in sorted(os.listdir(MATLAB_DIR)):
        if f.endswith(".m"):
            yield f, "\n".join(ln.split("%")[0] for ln in open(os.path.join(MATLAB_DIR, f)))


def test_matlab_glue_only_reads_members_the_reference_classes_have():
    """Every `self.<name>` / `mdl.<name>` / `m.<name>` the shipped .m files read must be a property or method of the
    reference's classes (EncounterModel, UncorEncounterModel, CorTerminalModel) -- round 1's glue read
    parameters_filename / isOverwriteZeroBoundaries / idxZeroBoundaries, which the objects do not keep
    (@EncounterModel/EncounterModel.m:98-104 are constructor locals)."""
    import re
    members = set(_upstream()["class_members"])
    assert {"G_initial", "N_transition", "dirichlet_initial", "start", "temporal_map", "r_initial", "n_initial",
            "boundaries", "resample_rates", "mdlFwd1_1", "dynLimits1", "bounds_sample"} <= members
    assert "parameters_filename" not in members and "idxZeroBoundaries" not in members
    seen = 0
    for f, src in _glue_sources():
        for obj, name in re.findall(r"\b(self|mdl|m)\.([A-Za-z]\w*)", src):
            assert name in members, "%s reads %s.%s, which the reference classes do not have" % (f, obj, name)
            seen += 1
    assert seen >= 30


def test_matlab_glue_calls_reference_functions_with_their_signatures():
    """The helper functions the glue calls must exist in the reference with the arity used."""
    import re
    up = _upstream()
    calls = {}
    for f, src in _glue_sources():
        src = src.replace("...\n", " ")
        for fn in up["function_arity"]:
            for m in re.finditer(r"\b%s\s*\(" % fn, src):
                depth, nargs = 1, 1
                for ch in src[m.end():]:
                    depth += {"(": 1, "[": 1, "{": 1, ")": -1, "]": -1, "}": -1}.get(ch, 0)
                    if depth == 0:
                        break
                    nargs += ch == "," and depth == 1
                calls.setdefault(fn, []).append(nargs)
    assert sorted(calls) == sorted(up["function_arity"])
    for fn, used in calls.items():
        assert set(used) == {up["function_arity"][fn]}, fn
    assert "EncounterModelEvents" in up["classes"]
    assert any(re.search(r"\bEncounterModelEvents\b", src) for _, src in _glue_sources())
