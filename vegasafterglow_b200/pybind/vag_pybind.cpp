// vag_pybind.cpp -- host C++ mirror of the reference's pybind11 surface for the model-evaluation
// path (module `VegasAfterglowC`, pybind/pybind.cpp:182-464), implemented on top of the C ABI
// include/vag.h.  Same factory / class / method / keyword names, same units, same error
// conventions (std::invalid_argument -> ValueError, wrong jet/medium type -> TypeError); the
// compute methods release the GIL like the reference (pybind.cpp:424-448).  Everything numeric
// happens in libvag_b200.so on the GPU: there is no host compute here.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <memory>
#include <mutex>
#include <optional>
#include <stdexcept>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/vag.h"

namespace py = pybind11;
using Real = double;

namespace {

[[noreturn]] void raise_for(int rc) {
    const std::string msg = vag_last_error();
    if (rc == VAG_ERR_INVALID) throw std::invalid_argument(msg);
    if (rc == VAG_ERR_UNSUPPORTED) {
        PyErr_SetString(PyExc_NotImplementedError, msg.c_str());
        throw py::error_already_set();
    }
    throw std::runtime_error(msg);
}
void check(int rc) {
    if (rc != VAG_OK) raise_for(rc);
}

// one context per device, shared by every Model of the process (calls are serialised per context)
struct Ctx {
    vag_context* h = nullptr;
    std::mutex mu;
    ~Ctx() {
        if (h) vag_destroy(h);
    }
};
std::shared_ptr<Ctx> context(int device) {
    static std::mutex mu;
    static std::vector<std::shared_ptr<Ctx>> table;
    std::lock_guard<std::mutex> lk(mu);
    if ((int)table.size() <= device) table.resize(device + 1);
    if (!table[device]) {
        auto c = std::make_shared<Ctx>();
        check(vag_create(device, &c->h));
        table[device] = c;
    }
    return table[device];
}

// ---- parameter carriers (the typed variants of JetVariant / MediumVariant) ----------------------
// Magnetar(L0, t0, q=2): pybind/pymodel.h:34-58, pybind/pybind.cpp:198-203
struct Magnetar {
    Real L0, t0, q;
    Magnetar(Real L0_, Real t0_, Real q_) : L0(L0_), t0(t0_), q(q_) {
        if (!(std::isfinite(L0) && L0 > 0)) throw std::invalid_argument("L0 must be finite and > 0");
        if (!(std::isfinite(t0) && t0 > 0)) throw std::invalid_argument("t0 must be finite and > 0");
        if (!(std::isfinite(q) && q > 0)) throw std::invalid_argument("q must be finite and > 0");
    }
    std::string repr() const {
        char buf[128];
        std::snprintf(buf, sizeof(buf), "Magnetar(L0=%g, t0=%g, q=%g)", L0, t0, q);
        return buf;
    }
};

struct Jet {
    int type;
    Real theta_c, E_iso, Gamma0, k_e, k_g, duration;
    bool spreading;
    Real theta_w{0.3}, E_iso_w{1e50}, Gamma0_w{50}, sigma0{0};
    bool has_magnetar{false};
    Real mag_L0{0}, mag_t0{0}, mag_q{0};
    std::string repr() const {
        char buf[200];
        static const char* names[] = {"TophatJet", "GaussianJet", "PowerLawJet", "TwoComponentJet", "StepPowerLawJet", "PowerLawWing"};
        const char* nm = names[type];
        snprintf(buf, sizeof(buf), "%s(theta_c=%.6g, E_iso=%.6g, Gamma0=%.6g)", nm, theta_c, E_iso, Gamma0);
        return buf;
    }
};
struct MediumP {
    int type;
    Real n_ism, A_star, n0;
    Real k_m{2};
};
struct Observer {
    Real lumi_dist, z, theta_obs, phi_obs;
};
struct Radiation {
    Real eps_e, eps_B, p, xi_e;
    bool ssc, kn;
};

void require(bool ok, const std::string& msg) {
    if (!ok) throw std::invalid_argument(msg);
}

Jet make_jet(int type, Real theta_c, Real E_iso, Real Gamma0, Real k_e, Real k_g, bool spreading, Real duration,
             const py::object& magnetar) {
    // pybind/pymodel.cpp:47-95
    require(std::isfinite(theta_c) && theta_c > 0 && theta_c <= 3.14159265358979323846 / 2, "theta_c must be in (0, pi/2]");
    require(std::isfinite(E_iso) && E_iso > 0, "E_iso must be finite and > 0");
    require(std::isfinite(Gamma0) && Gamma0 > 1.0, "Gamma0 must be > 1");
    require(std::isfinite(duration) && duration > 0, "duration must be finite and > 0");
    if (type == VAG_JET_POWERLAW || type == VAG_JET_STEP_POWERLAW || type == VAG_JET_POWERLAW_WING)
        require(std::isfinite(k_e) && k_e > 0 && std::isfinite(k_g) && k_g > 0, "k_e and k_g must be finite and > 0");
    Jet j{type, theta_c, E_iso, Gamma0, k_e, k_g, duration, spreading};
    if (!magnetar.is_none()) {
        const Magnetar mg = magnetar.cast<Magnetar>();
        j.has_magnetar = true;
        j.mag_L0 = mg.L0;
        j.mag_t0 = mg.t0;
        j.mag_q = mg.q;
    }
    return j;
}

struct Flux {
    py::object sync, ssc;
};
struct FluxDict {
    py::object total;
    Flux fwd, rvs;
};

py::array_t<double> empty0() { return py::array_t<double>(std::vector<py::ssize_t>{}); }

class Model {
  public:
    Model(py::object jet_obj, py::object medium_obj, Observer observer, Radiation fwd_rad, std::optional<Radiation> rvs_rad,
          std::optional<std::tuple<Real, Real, Real>> resolutions, Real rtol, bool axisymmetric, bool radiative_fireball,
          int device)
        : obs_(observer), fwd_(fwd_rad), rvs_(rvs_rad), device_(device) {
        if (!py::isinstance<Jet>(jet_obj)) throw py::type_error("jet must be TophatJet, GaussianJet, PowerLawJet, or Ejecta");
        if (!py::isinstance<MediumP>(medium_obj)) throw py::type_error("medium must be ISM, Wind, or Medium");
        const Jet jet = jet_obj.cast<Jet>();
        const MediumP med = medium_obj.cast<MediumP>();
        vag_params_default(&p_);
        p_.jet_type = jet.type;
        p_.spreading = jet.spreading;
        p_.theta_c = jet.theta_c;
        p_.E_iso = jet.E_iso;
        p_.Gamma0 = jet.Gamma0;
        p_.k_e = jet.k_e;
        p_.k_g = jet.k_g;
        p_.duration = jet.duration;
        p_.theta_w = jet.theta_w;
        p_.E_iso_w = jet.E_iso_w;
        p_.Gamma0_w = jet.Gamma0_w;
        p_.sigma0 = jet.sigma0;
        p_.has_magnetar = jet.has_magnetar ? 1 : 0;
        p_.magnetar_L0 = jet.mag_L0;
        p_.magnetar_t0 = jet.mag_t0;
        p_.magnetar_q = jet.mag_q;
        p_.medium_type = med.type;
        p_.n_ism = med.n_ism;
        p_.A_star = med.A_star;
        p_.n0 = med.n0;
        p_.wind_k_m = med.k_m;
        p_.lumi_dist = observer.lumi_dist;
        p_.z = observer.z;
        p_.theta_obs = observer.theta_obs;
        p_.phi_obs = observer.phi_obs;
        p_.fwd = vag_radiation{fwd_rad.eps_e, fwd_rad.eps_B, fwd_rad.p, fwd_rad.xi_e, fwd_rad.ssc, fwd_rad.kn};
        p_.has_rvs = rvs_rad ? 1 : 0;
        if (rvs_rad) p_.rvs = vag_radiation{rvs_rad->eps_e, rvs_rad->eps_B, rvs_rad->p, rvs_rad->xi_e, rvs_rad->ssc, rvs_rad->kn};
        p_.axisymmetric = axisymmetric;
        p_.radiative_fireball = radiative_fireball;
        // pybind/pymodel.h:633-647
        require(std::isfinite(rtol) && rtol > 0 && rtol < 1, "rtol must be in (0, 1), got " + std::to_string(rtol));
        p_.rtol = rtol;
        if (resolutions) {
            std::tie(p_.phi_resol, p_.theta_resol, p_.t_resol) = *resolutions;
            require(std::isfinite(p_.phi_resol) && p_.phi_resol > 0, "phi_resol must be finite and > 0");
            require(std::isfinite(p_.theta_resol) && p_.theta_resol > 0, "theta_resol must be finite and > 0");
            require(std::isfinite(p_.t_resol) && p_.t_resol > 0, "t_resol must be finite and > 0");
        }
        check(vag_params_validate(&p_));
    }

    FluxDict flux_density_grid(py::array_t<double, py::array::c_style | py::array::forcecast> t,
                               py::array_t<double, py::array::c_style | py::array::forcecast> nu) {
        const size_t n_t = t.size(), n_nu = nu.size();
        require(n_t > 0, "time array must be non-empty");
        require(n_nu > 0, "frequency array must be non-empty");
        std::vector<double> out(VAG_NCOMP * n_nu * n_t);
        {
            py::gil_scoped_release rel;
            auto ctx = context(device_);
            std::lock_guard<std::mutex> lk(ctx->mu);
            check(vag_flux_density_grid(ctx->h, &p_, 1, t.data(), n_t, nu.data(), n_nu, out.data(), nullptr));
        }
        return pack(out, {(py::ssize_t)n_nu, (py::ssize_t)n_t});
    }

    FluxDict flux_density(py::array_t<double, py::array::c_style | py::array::forcecast> t,
                          py::array_t<double, py::array::c_style | py::array::forcecast> nu) {
        const size_t n = t.size();
        require(n > 0, "time array must be non-empty");
        require(nu.size() > 0, "frequency array must be non-empty");
        require((size_t)nu.size() == n,
                "time and frequency arrays must have the same size\nIf you intend to get grid-like output, use the "
                "generic `flux_density_grid` instead");
        std::vector<double> out(VAG_NCOMP * n);
        {
            py::gil_scoped_release rel;
            auto ctx = context(device_);
            std::lock_guard<std::mutex> lk(ctx->mu);
            check(vag_flux_density_series(ctx->h, &p_, 1, t.data(), nu.data(), n, out.data(), nullptr));
        }
        return pack(out, {(py::ssize_t)n});
    }

    // PyModel::flux (pybind/pymodel.cpp:391-410)
    FluxDict flux(py::array_t<double, py::array::c_style | py::array::forcecast> t, double nu_min, double nu_max,
                  size_t num_nu) {
        const size_t n_t = t.size();
        require(n_t > 0, "time array must be non-empty");
        require(nu_min > 0, "nu_min must be positive");
        require(nu_max > nu_min, "nu_max must be greater than nu_min");
        require(num_nu >= 2, "num_nu must be at least 2");
        std::vector<double> out(VAG_NCOMP * n_t);
        {
            py::gil_scoped_release rel;
            auto ctx = context(device_);
            std::lock_guard<std::mutex> lk(ctx->mu);
            check(vag_flux_band(ctx->h, &p_, 1, t.data(), n_t, nu_min, nu_max, num_nu, out.data(), nullptr));
        }
        return pack(out, {(py::ssize_t)n_t});
    }

    // PyModel::flux_density_exposures (pybind/pymodel.cpp:412-496): sampling, evaluation and averaging on the GPU
    // (vag_flux_density_exposures checks the rest with the reference's messages)
    FluxDict flux_density_exposures(py::array_t<double, py::array::c_style | py::array::forcecast> t,
                                    py::array_t<double, py::array::c_style | py::array::forcecast> nu,
                                    py::array_t<double, py::array::c_style | py::array::forcecast> expo_time,
                                    size_t num_points) {
        const size_t n = t.size();
        require(n == (size_t)nu.size() && n == (size_t)expo_time.size(),
                "time, frequency, and exposure time arrays must have the same size");
        std::vector<double> out(VAG_NCOMP * n);
        {
            py::gil_scoped_release rel;
            auto ctx = context(device_);
            std::lock_guard<std::mutex> lk(ctx->mu);
            check(vag_flux_density_exposures(ctx->h, &p_, 1, t.data(), nu.data(), expo_time.data(), n, num_points,
                                             out.data(), nullptr));
        }
        return pack(out, {(py::ssize_t)n});
    }

    // Model.details (pybind/pymodel.cpp:315-348): assembled in Python from the device stage tables
    // (vegasafterglow_b200/details.py) -- broadcasting, unit conversion and the observer grids are host work
    py::object details(Real t_min, Real t_max) const {
        require(std::isfinite(t_min) && t_min > 0 && std::isfinite(t_max) && t_max > t_min, "need 0 < t_min < t_max");
        py::object engine = py::module_::import("vegasafterglow_b200.engine").attr("Engine")(device_);
        py::object dtype = py::module_::import("vegasafterglow_b200.abi").attr("PARAMS_DTYPE");
        py::bytes raw(reinterpret_cast<const char*>(&p_), sizeof(p_));
        py::object arr = py::module_::import("numpy").attr("frombuffer")(raw, dtype);
        return py::module_::import("vegasafterglow_b200.details").attr("simulation_details")(engine, arr, t_min, t_max);
    }

    const vag_params& params() const { return p_; }
    Observer obs_;
    Radiation fwd_;
    std::optional<Radiation> rvs_;

    std::string repr() const {
        char buf[256];
        snprintf(buf, sizeof(buf), "Model(observer=Observer(lumi_dist=%.6g, z=%.6g, theta_obs=%.6g), rtol=%.6g) [B200]",
                 obs_.lumi_dist, obs_.z, obs_.theta_obs, p_.rtol);
        return buf;
    }

  private:
    FluxDict pack(const std::vector<double>& out, std::vector<py::ssize_t> shape) const {
        size_t n = 1;
        for (auto s : shape) n *= (size_t)s;
        auto arr = [&](int comp) -> py::object {
            py::array_t<double> a(shape);
            std::copy(out.begin() + comp * n, out.begin() + (comp + 1) * n, a.mutable_data());
            return a;
        };
        // absent components are 0-d empty arrays, like default-constructed xt::xarray (pymodel.h:361-383)
        FluxDict f;
        f.total = arr(VAG_C_TOTAL);
        f.fwd.sync = arr(VAG_C_FWD_SYNC);
        f.fwd.ssc = fwd_.ssc ? arr(VAG_C_FWD_SSC) : py::object(empty0());
        f.rvs.sync = rvs_ ? arr(VAG_C_RVS_SYNC) : py::object(empty0());
        f.rvs.ssc = (rvs_ && rvs_->ssc) ? arr(VAG_C_RVS_SSC) : py::object(empty0());
        return f;
    }
    vag_params p_;
    int device_;
};

}  // namespace

PYBIND11_MODULE(VegasAfterglowC_b200, m) {
    m.doc() = "B200-native drop-in for the model-evaluation path of VegasAfterglowC (GPU only, no CPU fallback)";
    m.attr("fast_math_enabled") = false;
    m.attr("backend") = vag_version();

    py::class_<Jet>(m, "_Jet").def("__repr__", &Jet::repr);
    py::class_<Magnetar>(m, "Magnetar")
        .def(py::init<Real, Real, Real>(), py::arg("L0"), py::arg("t0"), py::arg("q") = 2)
        .def_readonly("L0", &Magnetar::L0)
        .def_readonly("t0", &Magnetar::t0)
        .def_readonly("q", &Magnetar::q)
        .def("__repr__", &Magnetar::repr);
    py::class_<MediumP>(m, "_Medium");

    m.def("TophatJet",
          [](Real theta_c, Real E_iso, Real Gamma0, bool spreading, Real duration, py::object magnetar) {
              return make_jet(VAG_JET_TOPHAT, theta_c, E_iso, Gamma0, 2, 2, spreading, duration, magnetar);
          },
          py::arg("theta_c"), py::arg("E_iso"), py::arg("Gamma0"), py::arg("spreading") = false, py::arg("duration") = 1,
          py::arg("magnetar") = py::none());
    m.def("GaussianJet",
          [](Real theta_c, Real E_iso, Real Gamma0, bool spreading, Real duration, py::object magnetar) {
              return make_jet(VAG_JET_GAUSSIAN, theta_c, E_iso, Gamma0, 2, 2, spreading, duration, magnetar);
          },
          py::arg("theta_c"), py::arg("E_iso"), py::arg("Gamma0"), py::arg("spreading") = false, py::arg("duration") = 1,
          py::arg("magnetar") = py::none());
    m.def("PowerLawJet",
          [](Real theta_c, Real E_iso, Real Gamma0, Real k_e, Real k_g, bool spreading, Real duration, py::object magnetar) {
              return make_jet(VAG_JET_POWERLAW, theta_c, E_iso, Gamma0, k_e, k_g, spreading, duration, magnetar);
          },
          py::arg("theta_c"), py::arg("E_iso"), py::arg("Gamma0"), py::arg("k_e"), py::arg("k_g"),
          py::arg("spreading") = false, py::arg("duration") = 1, py::arg("magnetar") = py::none());

    // Ejecta-family named factories (pybind/pybind.cpp:215-223, pybind/pymodel.cpp:97-146)
    auto gt1 = [](Real v, const char* nm) { require(std::isfinite(v) && v > 1.0, std::string(nm) + " must be > 1"); };
    auto pos = [](Real v, const char* nm) { require(std::isfinite(v) && v > 0, std::string(nm) + " must be finite and > 0"); };
    auto ang = [](Real v, const char* nm) {
        require(std::isfinite(v) && v > 0 && v <= 3.14159265358979323846 / 2, std::string(nm) + " must be in (0, pi/2]");
    };
    m.def("TwoComponentJet",
          [=](Real theta_c, Real E_iso, Real Gamma0, Real theta_w, Real E_iso_w, Real Gamma0_w, bool spreading, Real duration,
              py::object magnetar) {
              Jet j = make_jet(VAG_JET_TWO_COMPONENT, theta_c, E_iso, Gamma0, 2, 2, spreading, duration, magnetar);
              ang(theta_w, "theta_w");
              require(theta_w > theta_c, "theta_w (wing angle) must be greater than theta_c (core angle), got theta_w=" +
                                             std::to_string(theta_w) + ", theta_c=" + std::to_string(theta_c));
              pos(E_iso_w, "E_iso_w");
              gt1(Gamma0_w, "Gamma0_w");
              j.theta_w = theta_w;
              j.E_iso_w = E_iso_w;
              j.Gamma0_w = Gamma0_w;
              return j;
          },
          py::arg("theta_c"), py::arg("E_iso"), py::arg("Gamma0"), py::arg("theta_w"), py::arg("E_iso_w"), py::arg("Gamma0_w"),
          py::arg("spreading") = false, py::arg("duration") = 1, py::arg("magnetar") = py::none());
    m.def("StepPowerLawJet",
          [=](Real theta_c, Real E_iso, Real Gamma0, Real E_iso_w, Real Gamma0_w, Real k_e, Real k_g, bool spreading,
              Real duration, py::object magnetar) {
              Jet j = make_jet(VAG_JET_STEP_POWERLAW, theta_c, E_iso, Gamma0, k_e, k_g, spreading, duration, magnetar);
              pos(E_iso_w, "E_iso_w");
              gt1(Gamma0_w, "Gamma0_w");
              pos(k_e, "k_e");
              pos(k_g, "k_g");
              j.E_iso_w = E_iso_w;
              j.Gamma0_w = Gamma0_w;
              return j;
          },
          py::arg("theta_c"), py::arg("E_iso"), py::arg("Gamma0"), py::arg("E_iso_w"), py::arg("Gamma0_w"), py::arg("k_e"),
          py::arg("k_g"), py::arg("spreading") = false, py::arg("duration") = 1, py::arg("magnetar") = py::none());
    m.def("PowerLawWing",
          [=](Real theta_c, Real E_iso_w, Real Gamma0_w, Real k_e, Real k_g, bool spreading, Real duration) {
              Jet j = make_jet(VAG_JET_POWERLAW_WING, theta_c, 1.0, 2.0, k_e, k_g, spreading, duration, py::none());
              pos(E_iso_w, "E_iso_w");
              gt1(Gamma0_w, "Gamma0_w");
              pos(k_e, "k_e");
              pos(k_g, "k_g");
              j.E_iso_w = E_iso_w;
              j.Gamma0_w = Gamma0_w;
              return j;
          },
          py::arg("theta_c"), py::arg("E_iso_w"), py::arg("Gamma0_w"), py::arg("k_e"), py::arg("k_g"),
          py::arg("spreading") = false, py::arg("duration") = 1);
    // Extension (not a named factory of the reference, which needs Ejecta(sigma0=callable) for this):
    // a tophat jet with constant ejecta magnetisation sigma0.
    m.def("MagnetizedTophatJet",
          [](Real theta_c, Real E_iso, Real Gamma0, Real sigma0, bool spreading, Real duration) {
              Jet j = make_jet(VAG_JET_TOPHAT, theta_c, E_iso, Gamma0, 2, 2, spreading, duration, py::none());
              require(std::isfinite(sigma0) && sigma0 >= 0, "sigma0 must be finite and >= 0");
              j.sigma0 = sigma0;
              return j;
          },
          py::arg("theta_c"), py::arg("E_iso"), py::arg("Gamma0"), py::arg("sigma0"), py::arg("spreading") = false,
          py::arg("duration") = 1);

    m.def("ISM",
          [](Real n_ism) {
              require(std::isfinite(n_ism) && n_ism >= 0, "n_ism must be finite and >= 0");  // pymodel.cpp:148-151
              return MediumP{VAG_MEDIUM_ISM, n_ism, 0, INFINITY};
          },
          py::arg("n_ism"));
    m.def("Wind",
          [](Real A_star, std::optional<Real> n_ism, std::optional<Real> n0, Real k_m) {
              require(std::isfinite(A_star) && A_star > 0, "A_star must be finite and > 0");  // pymodel.cpp:153-186
              require(std::isfinite(k_m) && k_m > 0, "k_m must be finite and > 0");
              if (n_ism) require(std::isfinite(*n_ism) && *n_ism >= 0, "n_ism must be finite and >= 0");
              if (n0) require(*n0 > 0, "n0 must be > 0 (or +inf for no floor), got " + std::to_string(*n0));
              return MediumP{VAG_MEDIUM_WIND, n_ism.value_or(0), A_star, n0.value_or(INFINITY), k_m};
          },
          py::arg("A_star"), py::arg("n_ism") = py::none(), py::arg("n0") = py::none(), py::arg("k_m") = 2);

    py::class_<Observer>(m, "Observer")
        .def(py::init([](Real lumi_dist, Real z, Real theta_obs, Real phi_obs) {
                 // pybind/pymodel.h:190-204
                 require(std::isfinite(lumi_dist) && lumi_dist > 0, "lumi_dist must be finite and > 0");
                 require(std::isfinite(z) && z >= 0, "z must be finite and >= 0");
                 require(std::isfinite(theta_obs) && theta_obs >= 0 && theta_obs <= 3.14159265358979323846,
                         "theta_obs must be in [0, pi], got " + std::to_string(theta_obs));
                 require(std::isfinite(phi_obs), "phi_obs must be finite, got " + std::to_string(phi_obs));
                 return Observer{lumi_dist, z, theta_obs, phi_obs};
             }),
             py::arg("lumi_dist"), py::arg("z"), py::arg("theta_obs"), py::arg("phi_obs") = 0)
        .def_readonly("lumi_dist", &Observer::lumi_dist)
        .def_readonly("z", &Observer::z)
        .def_readonly("theta_obs", &Observer::theta_obs)
        .def_readonly("phi_obs", &Observer::phi_obs);

    py::class_<Radiation>(m, "Radiation")
        .def(py::init([](Real eps_e, Real eps_B, Real p, Real xi_e, bool ssc, bool kn) {
                 // pybind/pymodel.h:303-313
                 auto oi = [](Real v) { return std::isfinite(v) && v > 0 && v <= 1; };
                 require(oi(eps_e), "eps_e must be in (0, 1]");
                 require(oi(eps_B), "eps_B must be in (0, 1]");
                 require(oi(xi_e), "xi_e must be in (0, 1]");
                 require(std::isfinite(p) && p > 1.0, "p must be > 1");
                 return Radiation{eps_e, eps_B, p, xi_e, ssc, kn};
             }),
             py::arg("eps_e"), py::arg("eps_B"), py::arg("p"), py::arg("xi_e") = 1, py::arg("ssc") = false,
             py::arg("kn") = false)
        .def_readonly("eps_e", &Radiation::eps_e)
        .def_readonly("eps_B", &Radiation::eps_B)
        .def_readonly("p", &Radiation::p)
        .def_readonly("xi_e", &Radiation::xi_e)
        .def_readonly("ssc", &Radiation::ssc)
        .def_readonly("kn", &Radiation::kn);

    py::class_<Flux>(m, "Flux").def_readonly("sync", &Flux::sync).def_readonly("ssc", &Flux::ssc);
    py::class_<FluxDict>(m, "FluxDict")
        .def_readonly("total", &FluxDict::total)
        .def_readonly("fwd", &FluxDict::fwd)
        .def_readonly("rvs", &FluxDict::rvs);

    py::class_<Model>(m, "Model")
        .def(py::init<py::object, py::object, Observer, Radiation, std::optional<Radiation>,
                      std::optional<std::tuple<Real, Real, Real>>, Real, bool, bool, int>(),
             py::arg("jet"), py::arg("medium"), py::arg("observer"), py::arg("fwd_rad"), py::arg("rvs_rad") = py::none(),
             py::arg("resolutions") = py::none(), py::arg("rtol") = 1e-6, py::arg("axisymmetric") = true,
             py::arg("radiative_fireball") = true, py::arg("device") = 0)
        .def("flux_density_grid", &Model::flux_density_grid, py::arg("t"), py::arg("nu"))
        .def("flux_density", &Model::flux_density, py::arg("t"), py::arg("nu"))
        .def("flux", &Model::flux, py::arg("t"), py::arg("nu_min"), py::arg("nu_max"), py::arg("num_nu"))
        .def("flux_density_exposures", &Model::flux_density_exposures, py::arg("t"), py::arg("nu"), py::arg("expo_time"),
             py::arg("num_points") = 10)
        .def_property_readonly("observer", [](const Model& mdl) { return mdl.obs_; })
        .def_property_readonly("fwd_rad", [](const Model& mdl) { return mdl.fwd_; })
        .def_property_readonly("rvs_rad", [](const Model& mdl) { return mdl.rvs_; })
        .def_property_readonly("rtol", [](const Model& mdl) { return mdl.params().rtol; })
        // PyModel::get_resolutions (pybind/pybind.cpp:453, pymodel.h:750): the values in effect, i.e. an omitted
        // `resolutions` reads back as the defaults the constructor selected (pymodel.h:633-640)
        .def_property_readonly("resolutions",
                               [](const Model& mdl) {
                                   const vag_params& p = mdl.params();
                                   const bool r = p.has_rvs != 0;
                                   return std::make_tuple(p.phi_resol > 0 ? p.phi_resol : 0.06,
                                                          p.theta_resol > 0 ? p.theta_resol : (r ? 0.2 : 0.15),
                                                          p.t_resol > 0 ? p.t_resol : (r ? 10.0 : 6.0));
                               })
        .def_property_readonly("axisymmetric", [](const Model& mdl) { return mdl.params().axisymmetric != 0; })
        .def_property_readonly("radiative_fireball", [](const Model& mdl) { return mdl.params().radiative_fireball != 0; })
        .def_property_readonly("params_bytes",
                               [](const Model& mdl) { return py::bytes(reinterpret_cast<const char*>(&mdl.params()), sizeof(vag_params)); })
        .def("details", &Model::details, py::arg("t_min"), py::arg("t_max"))
        .def("__repr__", &Model::repr);
}
