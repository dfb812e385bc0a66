// Host driver: the B200 counterpart of the reference's main_run_job.cpp.  Same job structure -- parameters,
// init (default state or checkpoint restart), NaN check, time loop with print/plot cadence, checkpoint, run-time
// print, equilibrium extraction at kBT = 0 -- but the parameters come from a real input file, the solver calls go
// through the C ABI (include/bflbm.h) to the CUDA path, and the MultiFabs are device resident.
//
//   bflbm_run_job <Parameters file> [key=value ...]      (trailing key=value pairs override the file)
//
// File names follow main_run_job.cpp:150-202 (plot_file_dir, lbm_data_shshan_alpha0_.._xi_.._size.., f_checkpoint..).
// Structure factors (FHDeX StructFact in the reference, main_run_job.cpp:299-310, 330, 342-349, 50-54): accumulated on the
// GPU by libbflbm_sf.so (include/bflbm_sf.h) every out_SF_step steps inside the last plot_SF_window steps and written as
// <plot_file_root>_SF<step> at the last step.  Droplet runs print the centre of mass, the covariance eigenvalues and (if_print_radius)
// the fitted (W, R) of the tanh profile at every plot step, all reduced on the GPU(s).
#include <chrono>
#include <cstdarg>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <memory>
#include <sstream>

#include "../../../include/bflbm_sf.h"
#include "bflbm.hpp"
#include "parameters.hpp"
#include "plotfile.hpp"

using namespace bflbm;

static std::string fmt(const char* f, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, f);
  vsnprintf(buf, sizeof buf, f, ap);
  va_end(ap);
  return buf;
}

int main(int argc, char** argv) {
  if (argc < 2) {
    std::fprintf(stderr, "usage: %s <Parameters file> [key=value ...]\n", argv[0]);
    return 2;
  }
  try {
    std::stringstream text;
    {
      std::ifstream in(argv[1]);
      if (!in) throw std::runtime_error(std::string("cannot open ") + argv[1]);
      text << in.rdbuf() << '\n';
      for (int i = 2; i < argc; ++i) text << argv[i] << '\n';
    }
    const RunParameters R = parse_parameters(text);
    const bool noiseSwitch = R.kBT != 0.;  // main_run_job.cpp:63
    const auto t_start = std::chrono::steady_clock::now();

    bflbm_params p = default_params();
    p.kBT = R.kBT; p.tau_f = R.tau_f; p.tau_g = R.tau_g; p.alpha0 = R.alpha0; p.alpha1 = R.alpha1; p.kappa = R.kappa;
    p.rho_lo = R.rho_lo; p.rho_hi = R.rho_hi; p.seed = R.seed; p.step0 = R.step_continue;
    const int nx = R.nx, ny = R.ny, nz = R.nz;
    std::printf("%s\n", bflbm_version());
    std::printf("system = %s, box = %d x %d x %d, alpha0 = %g, kBT = %g, tau_f = %g, tau_g = %g\n", R.system.c_str(), nx, ny, nz, R.alpha0, R.kBT, R.tau_f, R.tau_g);
    if (R.plot_SF_window == 0) std::printf("plot_SF_window = 0 and No stuct factor will be calculated\n");

    // ---- file names, main_run_job.cpp:150-202 --------------------------------------------------------
    std::string plot_file_dir;
    if (R.system == "flat_interface") plot_file_dir = fmt("data_interface_alpha0_%.2f", R.alpha0);
    else if (R.system == "droplet") plot_file_dir = fmt("data_droplet_density_%.2f_alpha0_%.2f_r%.3f_size%d-%d-%d", R.rho_hi, R.alpha0, R.radius, nx, ny, nz);
    else plot_file_dir = std::string("data_mixture") + (R.plot_fields == "hydrovars" ? "_hydrovars" : "_lb_hydrovars");
    const std::string size_tag = fmt("_size%d-%d-%d", nx, ny, nz);
    const std::string base = R.root_path + "/" + plot_file_dir;
    const std::string plot_file_root = base + fmt("/lbm_data_shshan_alpha0_%.2f_xi_%.1e", R.alpha0, R.kBT) + size_tag + (noiseSwitch ? "_continue/plt" : "/plt");
    auto chk_name = [&](const char* which, int step, double temp) {
      return concatenate(base + "/" + which + "_checkpoint", step, R.Ndigits) + fmt("_alpha0_%.2f_xi_%.1e", R.alpha0, temp) + size_tag;
    };
    auto eq_name = [&](const char* which) { return base + "/equilibrium_" + which + fmt("_alpha0_%.2f", R.alpha0) + size_tag; };

    Lattice L(p, nx, ny, nz, R.device, R.ngpus, R.brick_lz);
    if (R.ngpus > 1) std::printf("%d GPUs: z-slabs, peer-to-peer ghost exchange\n", L.ngpus());

    // ---- fluctuating run on the equilibrium reference state, main_run_job.cpp:214-236 + LBM_binary.H:12, 92-107 -------
    if (noiseSwitch && R.use_ref_state) {
      std::printf("Noise switch on\n");
      const PlotfileData Er = read_plotfile(eq_name("rho")), Ep = read_plotfile(eq_name("phi")), Et = read_plotfile(eq_name("rhot"));
      for (const PlotfileData* E : {&Er, &Ep, &Et})
        if (E->nx != nx || E->ny != ny || E->nz != nz || E->ncomp != 1) throw std::runtime_error("equilibrium state does not match the box");
      auto total = [](const std::vector<double>& v) { double s = 0.; for (double x : v) s += x; return s; };
      std::printf("Mass rho_eq = %.15g\nMass phi_eq = %.15g\nMass rhot_eq = %.15g\n", total(Er.data), total(Ep.data), total(Et.data));
      // one GPU: the whole-box call (two-pass kernels); several: every slab on the brick kernel, centre of mass exchanged per step
      if (L.handle()) check(bflbm_set_reference_state(L.handle(), Er.data.data(), Ep.data.data(), Et.data.data()));
      else mcheck(bflbm_multi_set_reference_state(L.multi(), Er.data.data(), Ep.data.data(), Et.data.data()));
      double c[3];
      check(bflbm_get_reference_com(bflbm_multi_slab(L.multi(), 0), c));
      std::printf("Center of Mass: (%g,%g,%g)\n", c[0], c[1], c[2]);
    } else if (!noiseSwitch) {
      std::printf("Noise switch off, calculating the equilibrium state solutions...\n");
    }

    // ---- initialise, main_run_job.cpp:245-292 ------------------------------------------------------------
    if (R.if_continue_from_last_frame) {
      const double chk_temp = R.continueFromNonFluct ? 0. : R.kBT;
      std::printf("Loading in last frame checkpoint files....\n");
      const PlotfileData F = read_plotfile(chk_name("f", R.step_continue, chk_temp));
      const PlotfileData G = read_plotfile(chk_name("g", R.step_continue, chk_temp));
      if (F.nx != nx || F.ny != ny || F.nz != nz || F.ncomp != BFLBM_NVEL) throw std::runtime_error("checkpoint does not match the box");
      LBM_init(L, F.data, G.data);
    } else if (R.system == "mixture") {
      std::printf("Init mixture system ...\n");
      LBM_init_mixture(L);
    } else if (R.system == "flat_interface") {
      std::printf("Init flate interface system ...\n");
      LBM_init_stripe(R.init_frac, L);
    } else {
      std::printf("Init droplet system ...\n");
      LBM_init_droplet(R.radius, L);
    }
    std::printf("check initial hydrodynamic quantities validity ...\n");
    MultiFabNANCheck(L);  // main_run_job.cpp:294-297 (throws instead of exit(0))

    const bool plot_real = R.plot_fields == "hydrovars";
    // WriteOutput, main_run_job.cpp:35-55.  The frame is downloaded here; the file is written by the writer thread while the
    // main thread queues the next interval's steps (async_output = 0: inline, like the reference)
    FrameWriter writer(R.async_output);
    auto write_output = [&](int step) {
      const std::string dir = concatenate(plot_file_root, step, R.Ndigits);
      const int nc = plot_real ? BFLBM_NHYDRO : BFLBM_NHYDRO_BAR;
      auto frame = std::make_shared<std::vector<double>>(plot_real ? L.hydrovars() : L.hydrovars_bar());
      writer.push([=] { write_plotfile(dir, *frame, nc, nx, ny, nz, VariableNames(nc), step, step); });
    };
    if (R.plot_int > 0 && R.step_continue == 0) write_output(0);
    std::printf("LB initialized with alpha0 = %g and T = %g\n", R.alpha0, R.kBT);

    // ---- StructFact set-up, main_run_job.cpp:299-310 (pairs over hydrovs; only with noise and a window) -----------
    const int plot_SF = noiseSwitch ? R.plot_SF_window : 0;  // main_run_job.cpp:102
    const int SF_start = R.step_continue + R.nsteps - R.plot_SF_window;  // main_run_job.cpp:330
    const std::vector<int> pairA = {0, 1, 0, 2, 3, 4, 6, 7, 8, 2, 9, 15, 16, 17, 15, 18, 19, 20, 21, 20, 20, 21};
    const std::vector<int> pairB = {0, 1, 1, 2, 3, 4, 6, 7, 8, 6, 9, 15, 16, 17, 16, 18, 19, 20, 21, 21, 18, 18};
    bflbm_sf* structFact = nullptr;
    if (plot_SF > 0 && R.out_SF_step > 0 &&
        bflbm_sf_create_multi(L.multi(), (int)pairA.size(), pairA.data(), pairB.data(), nullptr, &structFact))
      throw std::runtime_error("structure-factor accumulator: creation failed");

    // ---- time loop, main_run_job.cpp:329-387 ------------------------------------------------------------------
    std::vector<double> radius_frames;  // main_run_job.cpp:112, 368
    const auto t_loop = std::chrono::steady_clock::now();
    const int last = R.step_continue + R.nsteps;
    int step = R.step_continue;
    while (step < last) {
      // run up to the next step at which the host has to look at the state
      int next = last;
      auto upto = [&](int interval) {
        if (interval > 0) next = std::min(next, (step / interval + 1) * interval);
      };
      upto(R.print_int);
      upto(R.plot_int);
      if (noiseSwitch) upto(R.out_noise_step);
      if (structFact) upto(R.out_SF_step);
      LBM_timestep(L, next - step);
      step = next;
      if (structFact && step >= SF_start && step % R.out_SF_step == 0 && bflbm_sf_accumulate(structFact))  // FortStructure(hydrovs, 0)
        throw std::runtime_error("structure-factor accumulator: accumulate failed");
      if (R.print_int > 0 && step % R.print_int == 0) std::printf("LB step %d info:\n", step);
      if (noiseSwitch && R.out_noise_step > 0 && step % R.out_noise_step == 0) {  // WriteOutNoise, Debug.H:380-409
        auto nz2 = std::make_shared<std::pair<std::vector<double>, std::vector<double>>>(L.noise());
        std::vector<std::string> fa, ga;
        for (int a = 0; a < BFLBM_NVEL; ++a) { fa.push_back("fa" + std::to_string(a)); ga.push_back("ga" + std::to_string(a)); }
        const std::string fdir = concatenate(plot_file_root + "_fnoise", step, R.Ndigits), gdir = concatenate(plot_file_root + "_gnoise", step, R.Ndigits);
        writer.push([=] {
          write_plotfile(fdir, nz2->first, BFLBM_NVEL, nx, ny, nz, fa, step, step);
          write_plotfile(gdir, nz2->second, BFLBM_NVEL, nx, ny, nz, ga, step, step);
        });
      }
      if (R.plot_int > 0 && step % R.plot_int == 0) {
        std::printf("\t**************************************\t\n\tLB step %d & Output\n\t**************************************\t\n", step);
        if (R.system == "droplet") {
          const auto c = update_com(L);
          std::printf("Center of Mass: (%g,%g,%g)\n", c[0], c[1], c[2]);
          const auto ev = fittingDropletCovariance(L);  // LBM_hydrovs.H:258-335 (shape-mode diagnostics)
          std::printf("Covariance eigenvalues: (%.10g,%.10g,%.10g)\n", ev[0], ev[1], ev[2]);
          if (R.if_print_radius) {  // main_run_job.cpp:364-368: fittingDropletParams(func_rho, 20, 0.01, 400, kappa, radius)
            double wr[3];
            int converged = 0;
            mcheck(bflbm_multi_fit_droplet(L.multi(), 20, 0.01, 400, R.kappa, R.radius, 0.2, 0.2, 0.02, wr, &converged));
            if (!converged) std::printf("statistical undulation %.2e out of bounds!\n", wr[2]);
            std::printf("fitting parameters for equilibrium density rho: (W=%f, R=%f)\n", wr[0], wr[1]);
            radius_frames.push_back(wr[1]);
          }
        }
        if (step >= R.out_step && step != last) write_output(step);
      }
      if (step == last) {
        write_output(step);
        if (structFact && bflbm_sf_samples(structFact) > 0) {  // structFact.WritePlotFile(step, time, root + "_SF", zero_avg = 1)
          std::vector<double> re(pairA.size() * L.cells());
          if (bflbm_sf_get(structFact, 1, re.data(), nullptr)) throw std::runtime_error("structure-factor accumulator: get failed");
          const std::vector<std::string> hn = VariableNames(BFLBM_NHYDRO);
          std::vector<std::string> names;
          for (size_t q = 0; q < pairA.size(); ++q) names.push_back("struct_fact_real_" + hn[pairA[q]] + "_" + hn[pairB[q]]);
          write_plotfile(concatenate(plot_file_root + "_SF", step, R.Ndigits), re, (int)pairA.size(), nx, ny, nz, names, step, step);
          std::printf("structure factor: %lld samples written\n", bflbm_sf_samples(structFact));
        }
      }
    }
    if (structFact) bflbm_sf_destroy(structFact);
    L.sync();
    writer.drain();  // every frame is on disk (the equilibrium extraction below reads them back)
    const double loop_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_loop).count();

    // ---- checkpoint, main_run_job.cpp:398-409 ---------------------------------------------------------------------
    {
      auto fg = L.populations();
      write_plotfile(chk_name("f", last, R.kBT), fg.first, BFLBM_NVEL, nx, ny, nz, {"rho_chk"}, 0, 0);
      write_plotfile(chk_name("g", last, R.kBT), fg.second, BFLBM_NVEL, nx, ny, nz, {"phi_chk"}, 0, 0);
    }
    MultiFabNANCheck(L);
    const double run_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_start).count();
    std::printf("Run time = %g\n", run_s);  // main_run_job.cpp:418-420
    std::printf("time loop: %d steps in %g s = %.1f MLUPS (incl. output)\n", R.nsteps, loop_s, (double)L.cells() * R.nsteps / loop_s / 1e6);

    // ---- equilibrium state = ensemble mean of the saved frames, main_run_job.cpp:422-439 / Debug.H:275-358 -------
    if (!noiseSwitch && R.plot_int > 0) {
      const int step1 = last - R.t_window, step2 = last;
      const int comp_of[3] = {0, 1, 5};  // rho, phi, rho+phi
      const char* nm[3] = {"rho", "phi", "rhot"};
      std::vector<std::vector<double>> mean(3, std::vector<double>(L.cells(), 0.));
      int frames = 0;
      for (int s = std::max(step1, R.out_step); s <= step2; s += R.plot_int) {
        if (s % R.plot_int != 0) continue;
        PlotfileData F;
        try { F = read_plotfile(concatenate(plot_file_root, s, R.Ndigits)); } catch (const std::exception&) { continue; }
        for (int k = 0; k < 3; ++k)
          for (size_t i = 0; i < L.cells(); ++i) mean[k][i] += F.data[(size_t)comp_of[k] * L.cells() + i];
        ++frames;
      }
      if (frames > 0) {
        for (int k = 0; k < 3; ++k)
          for (auto& v : mean[k]) v /= frames;
        // PrintConvergence, p_tag = 1 (Debug.H:275-358): lattice mean of the frame-averaged |frame - ensemble mean|
        std::vector<double> dev(3, 0.);
        for (int s = std::max(step1, R.out_step); s <= step2; s += R.plot_int) {
          if (s % R.plot_int != 0) continue;
          PlotfileData F;
          try { F = read_plotfile(concatenate(plot_file_root, s, R.Ndigits)); } catch (const std::exception&) { continue; }
          for (int k = 0; k < 3; ++k) {
            double a = 0.;
            for (size_t i = 0; i < L.cells(); ++i) a += std::fabs(F.data[(size_t)comp_of[k] * L.cells() + i] - mean[k][i]);
            dev[k] += a;
          }
        }
        std::printf("Convergence test emsemble selection: from step %d to step %d with step interval %d\n", std::max(step1, R.out_step), step2, R.plot_int);
        for (int k = 0; k < 3; ++k) {
          std::printf("convergence L1 (%s): %.6e\n", nm[k], dev[k] / frames / (double)L.cells());
          write_plotfile(eq_name(nm[k]), mean[k], 1, nx, ny, nz, {std::string(nm[k]) + "_eq"}, 0, 0);
        }
        std::printf("equilibrium state: mean of %d frames in steps [%d, %d]\n", frames, step1, step2);
      }
    }
    return 0;
  } catch (const std::exception& e) {
    std::fprintf(stderr, "bflbm_run_job: %s\n", e.what());
    return 1;
  }
}
