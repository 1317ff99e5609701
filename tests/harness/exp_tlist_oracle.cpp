// exp_tlist_oracle.cpp — the C++ restatement of the exponential solvers (oracle/vecode_oracle.cpp, orc_exp_ensemble) driven
// through a caller's ODEData.t_list (ode.rs:89, a pub field) instead of ODEData::new's [t0, tf] (ode.rs:144), keeping the state x
// of every system at each of its Chkpt / End events (ode.rs:165-176, 192-195) and the event of every call.
//
// TEST INFRASTRUCTURE ONLY (tests/_exp_tlist.py compiles it into a temporary directory). It includes the oracle's source, so
// BasisSplit, cfm_exp, ODEData, ODEAdaptiveData and gen_coef are the oracle's own; the driver below is orc_exp_ensemble with the
// list, the snapshots and the event record added, and computes the same bits as orc_exp_ensemble for the default list.
#include "../../oracle/vecode_oracle.cpp"

extern "C" {

struct ExpTlistCfg {
    ExpCfg base;
    int32_t n_tlist;     // entries of t_list, 0 for [t0, tf]
    const double* t_list;
    double* snap;        // nullable: [n_tlist][N][n] complex, the state of every system at its Chkpt / End event for t_list[k]
    int8_t* events;      // nullable: [N][events_cap], the event of each of the first events_cap calls (EV_*); later slots are left alone
    int64_t events_cap;
};

void orc_exp_tlist_ensemble(const ExpTlistCfg* tcfg, const double* basis /*[M][n][n] complex interleaved*/, const double* gp,
                      int32_t M_gen /*number of basis matrices the generator uses (rest are commutator slots)*/,
                      const double* cs, int64_t N, double* psi, double* t_out, double* h_out, int64_t* acc_out,
                      int64_t* rej_out, int32_t n_threads) {
    const ExpCfg* cfg = &tcfg->base;
    const int n = cfg->n, M = cfg->M;
    auto work = [&](int64_t lo, int64_t hi) {
        BasisSplit sp;
        sp.init(n, M, reinterpret_cast<const cplx*>(basis));
        sp.taylor_deg = cfg->taylor_deg;
        ExpCfg gc = *cfg;
        gc.M = M_gen;
        for (int64_t i = lo; i < hi; ++i) {
            const double* gpi = gp + (size_t)i * (M_gen - 1) * 3;
            std::vector<cplx> x0(n);
            for (int r = 0; r < n; ++r) x0[r] = {psi[((size_t)i * n + r) * 2], psi[((size_t)i * n + r) * 2 + 1]};
            ODEData<cplx> dat(cfg->t0, cfg->tf, x0, cfg->h0);
            if (tcfg->n_tlist > 0) dat.t_list.assign(tcfg->t_list, tcfg->t_list + tcfg->n_tlist);  // the pub field, ode.rs:89
            ODEAdaptiveData ad(cfg->order);
            ad.alpha = cfg->alpha, ad.rtol = cfg->rtol, ad.min_dt = cfg->min_dt, ad.max_dt = cfg->max_dt;
            std::vector<cplx> dx(x0), k((size_t)M), tmp(n), tmp2(n);
            std::vector<std::vector<cplx>> va;
            int64_t acc = 0, rej = 0, calls = 0;
            const bool want_err = !cfg->no_adaptive;
            auto pad = [&](std::vector<cplx>& v) { v.resize((size_t)M, cplx{0.0, 0.0}); };
            auto try_step = [&](double dt) {
                const double t = dat.t;
                if (cfg->scheme == 0) {  // midpoint, magnus.rs:10-26
                    const double t_mid = t + dt * 0.5;
                    std::vector<cplx> l;
                    gen_coef(gc, gpi, t_mid, l), pad(l);
                    const cplx cdt = {dt, 0.0};
                    for (auto& e : l) e = e * cdt;
                    sp.map_exp(l.data(), dat.x.data(), dat.next_x.data());
                } else if (cfg->scheme == 1) {  // cfm_general with CFM4 tables, cfm.rs:43-100, 131-154
                    va.resize(2);
                    for (int q = 0; q < 2; ++q) gen_coef(gc, gpi, t + C_GAUSS_LEGENDRE_4[q] * dt, va[q]), pad(va[q]);
                    cfm_exp(sp, dat.x.data(), tmp.data(), dt, va, k, &CFM_R4_J2_GL[0], 2);        // row 0
                    cfm_exp(sp, tmp.data(), dat.next_x.data(), dt, va, k, &CFM_R4_J2_GL[2], 2);   // row 1
                    if (want_err) {                                                                // cfm.rs:83-97
                        cfm_exp(sp, dat.x.data(), dx.data(), dt, va, k, CFM_R2_J1_GL, 2);
                        for (int r = 0; r < n; ++r) dx[r] = dx[r] - dat.next_x[r];
                    }
                } else if (cfg->scheme == 3) {  // cfm_general with runtime tables, cfm.rs:43-100
                    const int kn = cfg->n_nodes;
                    va.resize((size_t)kn);
                    for (int q = 0; q < kn; ++q) gen_coef(gc, gpi, t + cfg->c[q] * dt, va[q]), pad(va[q]);   // :70-72
                    cfm_exp(sp, dat.x.data(), tmp.data(), dt, va, k, cfg->alpha_tab, kn);                      // :74-75
                    for (int i = 1; i < cfg->n_rows; ++i) {                                                    // :76-80
                        cfm_exp(sp, tmp.data(), tmp2.data(), dt, va, k, cfg->alpha_tab + (size_t)i * kn, kn);
                        std::swap(tmp, tmp2);
                    }
                    dat.next_x = tmp;                                                                          // :81
                    if (want_err && cfg->alpha_err_tab) {                                                      // :83-97
                        cfm_exp(sp, dat.x.data(), tmp.data(), dt, va, k, cfg->alpha_err_tab, kn);
                        for (int i = 1; i < cfg->n_rows_err; ++i) {
                            cfm_exp(sp, tmp.data(), tmp2.data(), dt, va, k, cfg->alpha_err_tab + (size_t)i * kn, kn);
                            std::swap(tmp, tmp2);
                        }
                        for (int r = 0; r < n; ++r) dx[r] = tmp[r] - dat.next_x[r];
                    }
                } else {  // magnus_42, magnus.rs:28-83
                    const double c_mid = 0.288675134594812882254574390251;
                    const double b1 = dt * 0.5;
                    const double b2 = dt * dt * -0.144337567297406441127287195125;
                    const double mid_t = t + b1;
                    std::vector<cplx> l0, l1, w2((size_t)M, cplx{0.0, 0.0}), w1, w;
                    gen_coef(gc, gpi, mid_t - c_mid * dt, l0), pad(l0);
                    gen_coef(gc, gpi, mid_t + c_mid * dt, l1), pad(l1);
                    // commutator(l0, l1) expanded on the basis through the structure tensor (magnus.rs:55)
                    for (int a = 0; a < M; ++a)
                        for (int bq = 0; bq < M; ++bq) {
                            const cplx ab = l0[a] * l1[bq];
                            for (int cq = 0; cq < M; ++cq) {
                                const double sc = cs[((size_t)a * M + bq) * M + cq];
                                if (sc != 0.0) w2[cq] = w2[cq] + cplx{ab.re * sc, ab.im * sc};
                            }
                        }
                    const cplx cb2 = {b2, 0.0}, cb1 = {b1, 0.0};
                    for (auto& e : w2) e = e * cb2;                                   // magnus.rs:56
                    w1 = l0;                                                           // magnus.rs:59
                    for (int q = 0; q < M; ++q) w1[q] = w1[q] + l1[q];                 // :60
                    for (auto& e : w1) e = e * cb1;                                    // :61
                    w = w1;
                    for (int q = 0; q < M; ++q) w[q] = w[q] + w2[q];                   // :65-66
                    sp.map_exp(w.data(), dat.x.data(), dat.next_x.data());            // :72,75
                    if (want_err) {                                                    // :76-79
                        sp.map_exp(w1.data(), dat.x.data(), dx.data());
                        for (int r = 0; r < n; ++r) dx[r] = dx[r] - dat.next_x[r];
                    }
                }
            };
            int st = ST_OK;
            while (st == ST_OK && (cfg->max_calls <= 0 || calls < cfg->max_calls)) {
                ++calls;
                double dt = 0.0;
                int ev = dat.step_size_of(dat.h, &dt);
                const double h = dat.h;
                if (ev == EV_STEP) {
                    dat.next_dt = dt;
                    try_step(dt);
                    if (cfg->adaptive) {  // ode.rs:311-334 with norm = 2-norm of dx
                        const std::vector<cplx>& nv = (cfg->literal_norm && cfg->scheme == 2) ? x0 : dx;  // magnus.rs:274-276 reads adaptive_dat.dx (= x0)
                        double nn = 0.0;
                        for (int r = 0; r < n; ++r) nn = nn + (nv[r].re * nv[r].re + nv[r].im * nv[r].im);
                        ad.dx_norm = std::sqrt(nn);
                        const double f_ = ad.rtol / ad.dx_norm;
                        const double fp = rmin(rmax(ad.step_size_mul(f_), 0.3), 2.0);
                        dat.update_step_size(rmin(rmax(fp * h, ad.min_dt), ad.max_dt));
                        if (f_ <= 1.0) ev = EV_REJECT;
                    }
                }
                if (tcfg->events && calls <= tcfg->events_cap) tcfg->events[(size_t)i * tcfg->events_cap + (calls - 1)] = (int8_t)ev;
                if (tcfg->snap && (ev == EV_CHKPT || ev == EV_END) && dat.tgt_t < dat.t_list.size())  // what current() shows at this event
                    for (int r = 0; r < n; ++r) {
                        double* o = tcfg->snap + (((size_t)dat.tgt_t * N + i) * n + r) * 2;
                        o[0] = dat.x[r].re, o[1] = dat.x[r].im;
                    }
                switch (ev) {
                    case EV_STEP: dat.advance(), ++acc; break;
                    case EV_CHKPT: dat.checkpoint_update(); break;
                    case EV_REJECT: ++rej; break;
                    case EV_END: dat.checkpoint_update(), st = ST_DONE; break;
                }
            }
            for (int r = 0; r < n; ++r) psi[((size_t)i * n + r) * 2] = dat.x[r].re, psi[((size_t)i * n + r) * 2 + 1] = dat.x[r].im;
            if (t_out) t_out[i] = dat.t;
            if (h_out) h_out[i] = dat.h;
            if (acc_out) acc_out[i] = acc;
            if (rej_out) rej_out[i] = rej;
        }
    };
    if (n_threads <= 1) {
        work(0, N);
        return;
    }
    std::vector<std::thread> pool;
    const int64_t chunk = (N + n_threads - 1) / n_threads;
    for (int w = 0; w < n_threads; ++w) {
        const int64_t lo = w * chunk, hi = std::min<int64_t>(N, lo + chunk);
        if (lo < hi) pool.emplace_back(work, lo, hi);
    }
    for (auto& th : pool) th.join();
}

}  // extern "C"
