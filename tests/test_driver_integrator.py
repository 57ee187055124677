"""The drivers' ``integrator=`` names: an unknown name is refused with ValueError before any device or file work (it used
to run the leapfrog in the QG drivers and the host-controller ode23 in SW_zero_background_raytracing).  CPU only."""
import pytest

from swraytracing_b200 import drivers


@pytest.fixture
def no_work(monkeypatch):
    """every device and file entry point a driver reaches before its packet loop fails the test when called"""
    def called(*a, **k):
        raise AssertionError("the driver started work before checking its integrator")
    for name in ("g2k_dev", "k2g_dev", "Engine", "QGFlow", "QG2Flow", "parse_data", "_frozen_flow_setup"):
        monkeypatch.setattr(drivers, name, called)
    monkeypatch.setattr(drivers.fieldio, "PacketFrameWriter", called)
    monkeypatch.setattr(drivers.fieldio, "read_field", called)


@pytest.mark.parametrize("name", ["ode23_devce", "rk4", "", "ODE23"])
def test_qg_drivers_refuse_an_unknown_integrator(no_work, tmp_path, name):
    with pytest.raises(ValueError, match="integrator"):
        drivers.qgsw_raytrace(32, 4, 2.0, 1.0, 0.0, 0.5, 1.0, 1.0, outdir=str(tmp_path), integrator=name)
    with pytest.raises(ValueError, match="integrator"):
        drivers.qg2layersw_raytrace(32, 4, 2.0, 1.0, 0.0, 0.5, 1.0, 1.0, outdir=str(tmp_path), integrator=name)


@pytest.mark.parametrize("name", ["ode23_devce", "leapfrog"])
def test_sw_zero_background_refuses_an_unknown_integrator(no_work, tmp_path, name):
    with pytest.raises(ValueError, match="integrator"):
        drivers.SW_zero_background_raytracing(run_log_file=str(tmp_path / "no_such_log"), nx=32, f=1.0, Cg=1.0,
                                              integrator=name)


def test_accepted_names():
    for name in ("ode23", "ode23_device", "ode23_packets", "leapfrog"):
        drivers._Integrator(name, "qgsw_raytrace")
    for name in ("ode23", "ode23_device", "ode23_packets"):
        drivers._Integrator(name, "SW_zero_background_raytracing", leapfrog=False)
