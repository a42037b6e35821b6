"""Malformed calls to every entry point of include/emb200.h that takes a model or options are refused with a fixed
(code, message), before anything reaches the device: no launch, and the same answer with or without a GPU."""
import ctypes as C

import numpy as np
import pytest

from em_model_manned_bayes_b200 import _lib as L
from em_model_manned_bayes_b200.model import EncounterModel
from em_model_manned_bayes_b200.sample2track import integrate_opts


def synthetic(n_vars, r):
    """n_vars independent initial variables of r bins, each with a dynamic copy in the transition network."""
    n = n_vars
    uniform = [np.ones((r, 1))] * n
    return EncounterModel.from_arrays(np.zeros((n, n)), [r] * n, uniform, np.zeros((2 * n, 2 * n)), [r] * (2 * n),
                                      [None] * n + uniform, [[k + 1, n + k + 1] for k in range(n)],
                                      resample_rates=np.zeros(n))


@pytest.fixture(scope="module")
def models(model_paths):
    return {"uncor": EncounterModel(model_paths["uncor_1200code_v2p1"]), "initial_only": EncounterModel(model_paths["terminal_v3_radar_encounter_model"]),
            "five_tv": synthetic(5, 2), "wide": synthetic(2, 65)}


def opts(mem=L.EMB_MEM_HOST):
    o = L.SampleOpts()
    L.lib().emb_sample_opts_init(C.byref(o))
    o.mem = mem
    return o


def dependent_preset(m):
    """options presetting one initial variable that has a parent, with the parent left free"""
    o = opts()
    p, i = map(int, np.argwhere(m.G_initial)[0])
    o.start[i] = 1
    return o


def iopts(m, **fields):
    """the model's own integration options, with `fields` overridden"""
    o = integrate_opts(m)
    for k, v in fields.items():
        setattr(o, k, v)
    return o


RNG = L.Rng(1, 0)
BUF = np.zeros(1 << 16)            # large enough for whatever a call could touch before refusing
P = BUF.ctypes.data
OFFSETS = np.zeros(65, dtype=np.int64)
HIST = L.TrackOut(hist_initial=P)
DENSE = L.TrackOut(bins=P)
ROWS = np.arange(12, dtype=np.int32)
LIMITS = (L.DynLimits * 2)()
ASYNC = L.EMB_MEM_DEVICE | L.EMB_MEM_ASYNC
NULL_ROW = (C.c_int32 * 12)(*([0] * 11 + [-1]))
NO_MODELS = L.TerminalModels()


def tracks(m, n, T, o, out=None):
    return L.lib().emb_sample_tracks(m._h, C.byref(RNG), n, T, C.byref(o), C.byref(out or L.TrackOut()))


def events(m, n, T, o, capacity=0, rows=None, init=None):
    return L.lib().emb_sample_track_events(m._h, C.byref(RNG), n, T, C.byref(o), capacity, rows, OFFSETS.ctypes.data,
                                           C.byref(init) if init else None, None)


def packed(m, n, T, o, capacity=0, words=None):
    return L.lib().emb_sample_track_events_packed(m._h, C.byref(RNG), n, T, C.byref(o), capacity, words, words,
                                                  OFFSETS.ctypes.data, None, None)


def xyz(m, o, io, out=None, xyz_buf=P, good=None):
    return L.lib().emb_sample_tracks_xyz(m._h, C.byref(RNG), 4, 8, C.byref(o), C.byref(io),
                                         C.byref(out) if out else None, xyz_buf, good)


def terminal(models, tmax_s=10.0, rows=ROWS.ctypes.data):
    return L.lib().emb_terminal_propagate(C.byref(models), C.byref(RNG), 4, P, 4, C.cast(rows, C.POINTER(C.c_int32)),
                                          tmax_s, LIMITS, C.byref(opts()), C.byref(L.TrajOut(P, P)))


E_ARG, E_LIMIT = L.EMB_E_ARG, L.EMB_E_LIMIT
lib = L.lib
CASES = {
    # initial states
    "initial/null model": (lambda M: lib().emb_sample_initial(None, C.byref(RNG), 4, C.byref(opts()), P, None, None),
                           E_ARG, "null or negative argument"),
    "initial/negative n": (lambda M: lib().emb_sample_initial(M["uncor"]._h, C.byref(RNG), -1, C.byref(opts()), P, None, None),
                           E_ARG, "null or negative argument"),
    "initial/null opts": (lambda M: lib().emb_sample_initial(M["uncor"]._h, C.byref(RNG), 4, None, P, None, None),
                          E_ARG, "null or negative argument"),
    "initial/dependent preset": (lambda M: lib().emb_sample_initial(M["uncor"]._h, C.byref(RNG), 4,
                                                                   C.byref(dependent_preset(M["uncor"])), P, None, None),
                                 E_ARG, "Attempt to preset a dependent variable"),
    "initial/host async": (lambda M: lib().emb_sample_initial(M["uncor"]._h, C.byref(RNG), 4,
                                                             C.byref(opts(L.EMB_MEM_HOST | L.EMB_MEM_ASYNC)), P, None, None),
                           E_ARG, "EMB_MEM_ASYNC goes with EMB_MEM_DEVICE"),
    "initial_f32/null values": (lambda M: lib().emb_sample_initial_f32(M["uncor"]._h, C.byref(RNG), 4, C.byref(opts()), P,
                                                                      None, None),
                                E_ARG, "values must not be null"),
    # dense tracks
    "tracks/T < 1": (lambda M: tracks(M["uncor"], 4, 0, opts()), E_ARG, "null or out-of-range argument"),
    "tracks/no transition network": (lambda M: tracks(M["initial_only"], 4, 8, opts()), E_ARG, "dynvar:empty"),
    "tracks/stream index": (lambda M: tracks(M["five_tv"], 4, 2 ** 31 - 1, opts()), E_LIMIT, "32-bit stream index"),
    "tracks/host async": (lambda M: tracks(M["uncor"], 4, 8, opts(L.EMB_MEM_HOST | L.EMB_MEM_ASYNC)),
                          E_ARG, "EMB_MEM_ASYNC goes with EMB_MEM_DEVICE"),
    "tracks/histograms over 64 bins": (lambda M: tracks(M["wide"], 4, 8, opts(), HIST), E_LIMIT, "hold 64 bins"),
    # event rows
    "events/dense outputs in init": (lambda M: events(M["uncor"], 4, 8, opts(), init=DENSE), E_ARG,
                                     "dense outputs and histograms belong to emb_sample_tracks"),
    "events/T > 65535": (lambda M: events(M["uncor"], 4, 1 << 18, opts()), E_LIMIT, "T <= 65535"),   # 2^18 with <= 7 variables
    "events/capacity without rows": (lambda M: events(M["uncor"], 4, 8, opts(), capacity=16), E_ARG,
                                     "null or out-of-range argument"),
    "events/async": (lambda M: events(M["uncor"], 4, 8, opts(ASYNC)), E_ARG, "EMB_MEM_ASYNC goes with EMB_MEM_DEVICE"),
    "packed/T > 1023": (lambda M: packed(M["uncor"], 4, 1024, opts()), E_LIMIT, "T <= 1023"),
    "packed/capacity without rows": (lambda M: packed(M["uncor"], 4, 8, opts(), capacity=16), E_ARG,
                                     "null or out-of-range argument"),
    "packed/async": (lambda M: packed(M["uncor"], 4, 8, opts(ASYNC)), E_ARG, "EMB_MEM_ASYNC goes with EMB_MEM_DEVICE"),
    # fused xyz and integration
    "xyz/histograms": (lambda M: xyz(M["uncor"], opts(), iopts(M["uncor"]), out=HIST), E_ARG, "histograms belong to emb_sample_tracks"),
    "xyz/async": (lambda M: xyz(M["uncor"], opts(ASYNC), iopts(M["uncor"])), E_ARG, "EMB_MEM_ASYNC is not supported"),
    "xyz/bad indices": (lambda M: xyz(M["uncor"], opts(), iopts(M["uncor"], idx_altitude=0)), E_ARG, "idx_altitude / idx_speed"),
    "xyz/no outputs": (lambda M: xyz(M["uncor"], opts(), iopts(M["uncor"]), xyz_buf=None), E_ARG, "xyz and is_good are both null"),
    "integrate/bad indices": (lambda M: lib().emb_tracks_integrate(M["uncor"]._h, 4, 8, P, P, C.byref(iopts(M["uncor"], idx_acceleration=1)), P, None),
                              E_ARG, "must be time-varying variables"),
    # terminal encounters
    "terminal/null model": (lambda M: terminal(NO_MODELS), E_ARG, "emb_terminal_models: null model"),
    "terminal/tmax_s": (lambda M: terminal(NO_MODELS, tmax_s=32767.0), E_ARG, "tmax_s must be in [0, 32767)"),
    "terminal/negative geo row": (lambda M: terminal(NO_MODELS, rows=C.addressof(NULL_ROW)), E_ARG, "geo_rows: negative row"),
    "screen/tmax_s": (lambda M: lib().emb_terminal_screen(P, P, 4, -1.0, 500.0, 100.0, C.byref(opts()),
                                                          C.byref(L.ScreenOut(P, P, P, P, P))),
                      E_ARG, "tmax_s must be in [0, 32767)"),
    # scoring
    "loglik_initial/async": (lambda M: lib().emb_loglik_initial(M["uncor"]._h, 4, P, C.byref(opts(ASYNC)), P, None),
                             E_ARG, "loglik: EMB_MEM_ASYNC is not supported"),
    "loglik_tracks/no transition network": (lambda M: lib().emb_loglik_tracks(M["initial_only"]._h, 4, 8, P, P, C.byref(opts()),
                                                                              P, P),
                                            E_ARG, "dynvar:empty"),
    "loglik_tracks/T < 1": (lambda M: lib().emb_loglik_tracks(M["uncor"]._h, 4, 0, P, P, C.byref(opts()), P, P),
                            E_ARG, "null or out-of-range argument"),
    # priors
    "set_prior/unknown kind": (lambda M: lib().emb_set_prior(M["uncor"]._h, 0, 7, 1.0), E_ARG, "prior:unknown"),
    "set_prior/stay on the initial network": (lambda M: lib().emb_set_prior(M["uncor"]._h, 0, L.EMB_PRIOR_STAY, 1.0), E_ARG,
                                              "stay prior applies to the transition network only"),
    "set_prior/negative": (lambda M: lib().emb_set_prior(M["uncor"]._h, 1, L.EMB_PRIOR_CONSTANT, -1.0), E_ARG,
                           "prior must be >= 0"),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_malformed_call_is_refused_before_any_launch(models, case):
    call, code, message = CASES[case]
    launches = lib().emb_launch_count()
    rc = call(models)
    err = lib().emb_last_error().decode()
    assert (rc, message in err) == (code, True), (rc, err)
    assert lib().emb_launch_count() == launches
