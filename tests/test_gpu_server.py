"""SURVEY 8(f) row 3: the reference's TCP front end (``OBE_Server``, optbayesexpt/obe_server.py:118-315, wire format
obe_socket.py:12-25,88-129) driving the GPU engine.  The server class is the UNMODIFIED reference's when it is installed
in baseline/_ref (baseline/install_reference.sh), else its restatement in oracle/obe_server.py; only the engine it is
told to make (``make_obe``) is ours.  The client speaks the reference's protocol (10-digit length + JSON) over loopback:
optset / goodset / newdat / getmean / getstd / getcov / getset / getcon / getpar / getwgt / ready / done.
Only getpar / getwgt may bring the cloud back to the host."""
import os
import socket
import sys
import threading
import warnings

import numpy as np
import pytest
from numpy.testing import assert_allclose

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _reference():
    path = os.path.join(ROOT, 'baseline', '_ref')
    if os.path.isdir(os.path.join(path, 'optbayesexpt')):
        if path not in sys.path:
            sys.path.insert(0, path)
        warnings.simplefilter('ignore', SyntaxWarning)
        import optbayesexpt
        return optbayesexpt
    from oracle import obe_server
    return obe_server


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def test_reference_server_drives_the_gpu_engine():
    ref = _reference()
    import optbayesexpt_b200 as obe
    from oracle.scenarios import build_inputs, by_name
    sc = by_name('c1_find_peak')
    inp = build_inputs(sc, 20000)
    port = _free_port()
    server = ref.OBE_Server(port=port)
    server.make_obe(obe.OptBayesExpt, ('lorentzian_hwhm', inp['setting_values'], inp['prior'], inp['cons']),
                    scale=False, default_noise_std=500.0, seed=3)
    eng = server.obe_engine
    assert isinstance(eng, obe.OptBayesExpt)
    errors = []

    def serve():
        try:
            import torch
            torch.cuda.set_device(0)
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                server.run()
        except Exception as exc:            # pragma: no cover
            errors.append(exc)
    th = threading.Thread(target=serve, daemon=True)
    th.start()
    client = ref.Socket('client', port=port)
    try:
        assert client.tcpcmd({'command': 'ready'}) == 'OK'
        sets = client.tcpcmd({'command': 'getset'})
        assert_allclose(np.array(sets), eng.allsettings)
        assert client.tcpcmd({'command': 'getcon'}) == list(inp['cons'])
        truth = (3.14, -1200.0, 50400.0)
        meas = np.random.default_rng(5)
        for it in range(12):
            cmd = {'command': 'optset'} if it % 3 else {'command': 'goodset', 'pickiness': 9}
            x = client.tcpcmd(cmd)
            assert len(x) == 1 and 1.5 <= x[0] <= 4.5
            y = truth[2] + truth[1] / (((x[0] - truth[0]) / 0.1) ** 2 + 1) + 500.0 * meas.standard_normal()
            assert client.tcpcmd({'command': 'newdat', 'x': x, 'y': [y], 's': [500.0]}) == 'OK'
            mean = np.array(client.tcpcmd({'command': 'getmean'}))
            std = np.array(client.tcpcmd({'command': 'getstd'}))
            cov = np.array(client.tcpcmd({'command': 'getcov'}))
            assert mean.shape == (3,) and std.shape == (3,) and cov.shape == (3, 3)
            assert_allclose(mean, eng.mean(), rtol=0, atol=0)
            assert_allclose(np.sqrt(np.diag(cov)), std, rtol=1e-3)      # np.cov normalisation vs biased std
            # none of the run-time commands brought the cloud back to the host
            assert eng._host_particles is None and eng._host_weights is None
        # the posterior moved towards the truth
        assert abs(mean[0] - truth[0]) < 3 * std[0] + 0.05
        par = np.array(client.tcpcmd({'command': 'getpar'}))
        assert par.shape == (3, 20000) and eng._host_particles is not None and eng._host_weights is None
        wgt = np.array(client.tcpcmd({'command': 'getwgt'}))
        assert wgt.shape == (20000,) and abs(wgt.sum() - 1.0) < 1e-12 and eng._host_weights is not None
        assert_allclose((par * wgt).sum(axis=1), mean, rtol=1e-10)
    finally:
        assert client.tcpcmd({'command': 'done'}) == 'OK'
        th.join(timeout=30)
        server.server.close()
    assert not errors, errors
    assert not th.is_alive()
