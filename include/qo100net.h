/*
 * qo100net.h -- C-ABI of libqo100net: B200-native (sm_100a) frequency-swept
 * evaluation of 2-port RF networks and component-tolerance Monte-Carlo yield.
 *
 * Drop-in boundary.  The reference tree (vankxr/qo-100-tools) has NO code, FFI
 * or plugin interface for this path: its util/ directory holds the inputs and
 * outputs of external GUI tools.  The boundary this library replaces is
 * therefore the *file formats* on the input side and Qucs-dataset-shaped
 * arrays on the output side; each entry point cites the reference artefact
 * (relative to the reference root) whose tool action it replaces.
 *
 * Conventions: every function returns 0 (QO_OK) or a negative qo_status and
 * never aborts.  All array arguments are HOST pointers owned by the caller
 * unless the name says "_dev"; the library does its own H2D / D2H.  Opaque
 * handles are owned by the library and released with the matching *_free /
 * *_destroy.  A qo_ctx is single-caller (not re-entrant); distinct contexts
 * are independent.  There is NO CPU fallback: compute entry points fail with
 * QO_ERR_NO_DEVICE when no CUDA device is usable.
 */
#ifndef QO100NET_H
#define QO100NET_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    QO_OK = 0,
    QO_ERR_ARG = -1,
    QO_ERR_IO = -2,
    QO_ERR_PARSE = -3,
    QO_ERR_UNSUPPORTED = -4,
    QO_ERR_NOMEM = -5,
    QO_ERR_NO_DEVICE = -6,
    QO_ERR_CUDA = -7,
    QO_ERR_NCCL = -8,
    QO_ERR_RANGE = -9
} qo_status;

typedef struct qo_net qo_net;   /* immutable element list + terminations */
typedef struct qo_ctx qo_ctx;   /* owns the device(s), stream(s), scratch buffers */
typedef struct qo_plan qo_plan; /* a Monte-Carlo job resident in HBM */
typedef struct { double re, im; } qo_c64;

/* ---- element list ------------------------------------------------------ */
typedef enum {
    QO_SER_R = 1, QO_SHUNT_R = 2,            /* p0 = R                                   */
    QO_SER_L = 3, QO_SHUNT_L = 4,            /* p0 = L, p1 = ESR, p2 = Cp  (Z=(R+jwL)||1/jwCp) */
    QO_SER_C = 5, QO_SHUNT_C = 6,            /* p0 = C, p1 = ESR, p2 = ESL (Z=R+jwLs+1/jwC)    */
    QO_SER_LC_SER = 7,                       /* p0 = L, p1 = C : Z = jwL + 1/(jwC)       */
    QO_SER_LC_PAR = 8,                       /*                 Z = 1/(jwC + 1/(jwL))    */
    QO_SHUNT_LC_SER = 9,                     /*                 Y = 1/(jwL + 1/(jwC))    */
    QO_SHUNT_LC_PAR = 10,                    /*                 Y = jwC + 1/(jwL)        */
    QO_TLINE = 11,                           /* p0 = Z0, p1 = angle[deg] at p2 = f0 (lossless) */
    QO_CPL_THRU = 12,                        /* coupled line, through path, far ports in Zt:
                                                p0=Z0e p1=Z0o p2=ang_e p3=ang_o [deg] p4=f0 p5=Zt */
    QO_SUBST = 13,                           /* p = er, h, t, tand, rho, D (Qucs SUBST)  */
    QO_MLIN = 14,                            /* p0 = W, p1 = L                           */
    QO_MCORN = 15,                           /* p0 = W                                   */
    QO_MTEE = 16,                            /* p0 = Wa, p1 = Wb, p2 = W2; opens the side arm:
                                                the following elements, junction outward, up to */
    QO_MOPEN = 17,                           /* p0 = W; open end closing the side arm    */
    QO_SBLOCK = 18,                          /* measured two-port (Touchstone): p0 = block index in the net,
                                                p1 = 1 polar / 0 rectangular interpolation (Qucs SPfile)   */
    QO_CPL_MS = 19                           /* PHYSICAL coupled microstrip, through path (far ports in Zt), on the
                                                preceding QO_SUBST (er, h, t): p0=W p1=S p2=L p3=H_t (cover height)
                                                p4=f0 (analysis frequency, as QucsTranscalc "Freq") p5=Zt.  Per
                                                sample the geometry / substrate draws go through the coupled-
                                                microstrip analysis (qo_cpl_analyze's model) to Z0e, Z0o, theta_e,
                                                theta_o, then the ideal coupled-line block: util/directional-
                                                couplers/ *.trc:6-20 with manufacturing tolerances on W, S, H, Er */
} qo_kind;
#define QO_NPARAM 6
typedef struct { int32_t kind; int32_t flags; double p[QO_NPARAM]; } qo_elem;

/* rf-tools.com LC-filter export (SVG).  Replaces the rf-tools analysis of
 * util/if-bandpass-filter/schematic.svg:174-217, util/gpsdo-ouput-filters/10M/
 * schematic.svg:174-231, docs/gpsdo-filters/{15M,40M,60M}.svg:174-241,
 * docs/upconverter/upconverter-lol-filter.svg:174-249. */
int qo_net_load_rftools_svg(const char *path, qo_net **out);
/* Qucs 0.0.19 schematic: components, properties, Eqn constants and the
 * cascade recovered from wire/pin coordinates.  Replaces the Qucs netlister
 * for util/pa-lpf-simulation/pa-lpf-simulation.sch:19-61 (2-port microstrip
 * cascades with MTEE side stubs ending in MOPEN). */
int qo_net_load_qucs_sch(const char *path, qo_net **out);
/* the .SP sweep of a Qucs schematic (pa-lpf-simulation.sch:59): type 0=lin 1=log */
int qo_qucs_sch_sweep(const char *path, int *type, double *f0, double *f1, int *n);
/* QucsTranscalc CoupledMicrostrip save file (util/directional-couplers/ *.trc:5-21).
 * phys (nullable) = { Er, H, H_t, T, W, S, L, Tand } in SI units. */
int qo_cpl_load_trc(const char *path, double *z0e, double *z0o, double *ang_deg, double *f0_hz, double phys[8]);
/* QucsTranscalc "analyze" for CoupledMicrostrip (physical -> electrical), the
 * action that produced *.trc:18-20.  SI units; angles in degrees. */
int qo_cpl_analyze(double w, double s, double h, double t, double er, double ht, double f, double len,
                   double *z0e, double *z0o, double *ang_e_deg, double *ang_o_deg);
/* QucsTranscalc "synthesize" for CoupledMicrostrip (electrical -> physical), the action that produced the W / S / L
 * lines *.trc:15-17 from Z0e / Z0o / Ang_l :18-20 (Ang_l = sqrt(theta_e theta_o)).  QO_ERR_RANGE when the substrate
 * cannot realise the pair. */
int qo_cpl_synthesize(double z0e, double z0o, double ang_deg, double h, double t, double er, double ht, double f,
                      double *w, double *s, double *len);

int qo_net_from_elements(const qo_elem *e, int n, double rs, double rl, qo_net **out);
/* pcb/generic-filter (README.md:13; qo-100-generic-filter.sch:1450-1488,1703-1995):
 * up-to-11th-order ladders, 6 series + 5 shunt branches, series first. */
int qo_net_cheby_lpf(int order, double ripple_db, double fc, double z0, int series_first, qo_net **out);
int qo_net_butter_lpf(int order, double fc, double z0, int series_first, qo_net **out);
/* ESR/SRF parasitics: L: R = wc*L/q_l, Cp s.t. SRF = srf_l_mult*fc;
 * C: ESR = esr_c, ESL s.t. SRF = srf_c_mult*fc (model evidenced by
 * util/pa-bias-simulation/pa-bias-simulation.sch:19-34 and the Coilcraft .s2p) */
int qo_net_add_parasitics(qo_net *net, double fc, double q_l, double srf_l_mult, double esr_c, double srf_c_mult);
int qo_net_concat(const qo_net *a, const qo_net *b, qo_net **out); /* a then b; terminations rs(a), rl(b) */
int qo_net_num_elements(const qo_net *net);
int qo_net_get_elements(const qo_net *net, qo_elem *out, int cap); /* returns count */
int qo_net_terminations(const qo_net *net, double *rs, double *rl);
/* free-text title lines found by the loader (e.g. "Cutoff Frequency = 15.00 MHz") */
const char *qo_net_title(const qo_net *net);
void qo_net_free(qo_net *net);

/* f_k = f0 + k*((f1-f0)/(n-1)) with no FMA -- bit-exact vs
 * util/pa-lpf-simulation/pa-lpf-simulation.dat:6-5005 */
int qo_grid_lin(double f0, double f1, int n, double *f);
int qo_grid_log(double f0, double f1, int n, double *f);

/* ---- Touchstone two-port blocks (Qucs "SPfile") ------------------------- */
/* The measured inductors the reference's bias schematics pull in with
 *   <SPfile ... "11SQ39N.S2P" ... "polar" "linear">  util/pa-bias-simulation/pa-bias-simulation.sch:39
 *   <SPfile ... "06HP47N.s2p" ... "polar" "linear">  util/preamp-bias-simulation/preamp-bias-simulation.sch:32
 * and docs/pa-driver/pa_20W_vdd_32V_idq_180mA.s2p.  Touchstone v1, 2 ports, "# HZ|KHZ|MHZ|GHZ S MA|DB|RI R z0". */
typedef struct qo_s2p qo_s2p;
int qo_s2p_load(const char *path, qo_s2p **out);
int qo_s2p_from_arrays(const double *f, int n, const qo_c64 *s11, const qo_c64 *s21, const qo_c64 *s12, const qo_c64 *s22,
                       double z0, qo_s2p **out);
int qo_s2p_num_points(const qo_s2p *blk);
double qo_s2p_z0(const qo_s2p *blk);
int qo_s2p_get(const qo_s2p *blk, double *f, qo_c64 *s11, qo_c64 *s21, qo_c64 *s12, qo_c64 *s22, int cap); /* returns n */
/* S at arbitrary frequencies: linear in f between the bracketing points, on (|S|, phase along the shorter arc)
 * when polar != 0 else on (re, im); the end segments are extrapolated linearly outside the measured range
 * (Qucs' behaviour: util/pa-bias-simulation/pa-bias-simulation.dat is reproduced only this way).  Host routine (the kernels
 * use the same routine at plan creation to build the per-frequency ABCD table of the block). */
int qo_s2p_interp(const qo_s2p *blk, const double *f, int nf, int polar, qo_c64 *s11, qo_c64 *s21, qo_c64 *s12, qo_c64 *s22);
/* least-squares fit of the ESR/SRF inductor model Z = (r0 + r1 sqrt(f) + jwL) || 1/(jwCp) to a block measured
 * in series between its ports, over [fmin, fmax]; srf and rms_rel nullable */
int qo_s2p_fit_inductor(const qo_s2p *blk, double fmin, double fmax, double *L, double *r0, double *r1, double *cp,
                        double *srf, double *rms_rel);
void qo_s2p_free(qo_s2p *blk);
/* a one-element network holding a copy of the block; combine with qo_net_concat */
int qo_net_from_sblock(const qo_s2p *blk, int polar, double rs, double rl, qo_net **out);

/* ---- N-port nodal analysis ------------------------------------------------ */
/* General linear networks that are not a 2-port cascade: the reference's bias networks
 * util/pa-bias-simulation/pa-bias-simulation.sch:19-72 (5 ports; R, C, ideal VCVS buffers :40,59, the measured
 * inductor via SPfile :39), whose Qucs result is util/pa-bias-simulation/pa-bias-simulation.dat:1-85035.
 * Modified nodal analysis per (sample, frequency) point on the GPU: one LU factorisation, one substitution
 * per port.  Node 0 is ground; ports are numbered 1.. in the order they are added. */
typedef struct qo_nodal qo_nodal;
typedef enum { QO_NB_R = 1, QO_NB_L = 2, QO_NB_C = 3, QO_NB_VCVS = 4, QO_NB_SBLOCK = 5 } qo_nb_kind;
/* R: node a,b p0=R | L: a,b p0=L p1=ESR p2=Cp | C: a,b p0=C p1=ESR p2=ESL  (same parasitic forms as QO_SER_L/C)
 * VCVS: node in+, out+, out-, in-; p0=gain p1=delay[s] | SBLOCK: node t1, t2, ref; p0=block index p1=polar p2=z0 */
typedef struct { int32_t kind; int32_t node[4]; double p[4]; } qo_branch;
int qo_nodal_create(int n_nodes, qo_nodal **out);
int qo_nodal_add_branch(qo_nodal *nd, const qo_branch *b);
int qo_nodal_add_port(qo_nodal *nd, int node, double z0);                 /* returns the port's number (1..) */
int qo_nodal_add_sblock(qo_nodal *nd, const qo_s2p *blk, int *index);     /* copies the block */
int qo_nodal_load_qucs_sch(const char *path, qo_nodal **out);             /* Qucs netlister for R, L, C, GND, Pac, VCVS, SPfile */
int qo_nodal_num_nodes(const qo_nodal *nd);
int qo_nodal_num_ports(const qo_nodal *nd);
int qo_nodal_num_branches(const qo_nodal *nd);
int qo_nodal_get_branches(const qo_nodal *nd, qo_branch *out, int cap);   /* returns count */
int qo_nodal_get_ports(const qo_nodal *nd, int *node, double *z0, int cap);
void qo_nodal_free(qo_nodal *nd);
/* compute entry points: qo_nodal_sweep / qo_nodal_mc_run below */

/* ---- Qucs dataset (.dat) reader / writer --------------------------------- */
/* The layout Qucs 0.0.19 writes for util/pa-lpf-simulation/pa-lpf-simulation.dat:1-35018:
 * "<indep NAME N>" / "<dep NAME INDEP>" blocks of "%+.20e" reals or "%+.20e+j%.20e" complex values.
 * qo_dat_read -> qo_dat_write reproduces that file byte for byte; qo_dat_from_sweep builds the dataset
 * Qucs would write for a 2-port .SP sweep with the dB() equations of pa-lpf-simulation.sch:59-60
 * (frequency, S11_dB, S21_dB, S[1,1], S[1,2], S[2,1], S[2,2]). */
typedef struct qo_dat qo_dat;
int qo_dat_create(qo_dat **out);
int qo_dat_read(const char *path, qo_dat **out);
int qo_dat_write(const qo_dat *dat, const char *path);
int qo_dat_add_indep(qo_dat *dat, const char *name, const double *v, int n);
int qo_dat_add_dep(qo_dat *dat, const char *name, const char *indep, const double *re, const double *im /* NULL = real */, int n);
int qo_dat_count(const qo_dat *dat);
/* variable i: name, the independent it hangs on ("" for an independent variable), points, complex? */
int qo_dat_info(const qo_dat *dat, int i, const char **name, const char **indep, int *n, int *is_complex);
/* copies up to cap values (im nullable); returns the variable's point count */
int qo_dat_get(const qo_dat *dat, const char *name, double *re, double *im, int cap);
int qo_dat_from_sweep(const double *f, int nf, const qo_c64 *s11, const qo_c64 *s12, const qo_c64 *s21, const qo_c64 *s22, qo_dat **out);
void qo_dat_free(qo_dat *dat);

/* ---- compute ----------------------------------------------------------- */
/* ngpus devices 0..ngpus-1 in ONE process (samples sharded, counters combined
 * by NCCL all-reduce when libnccl is loadable, see DESIGN.md).  One process
 * per GPU (torchrun) uses qo_ctx_create_on_device + qo_plan_launch with a
 * caller-owned device counter buffer that torch.distributed all-reduces. */
int qo_ctx_create(int ngpus, qo_ctx **out);
int qo_ctx_create_on_device(int device, qo_ctx **out);
int qo_ctx_set_stream(qo_ctx *ctx, void *cuda_stream); /* cudaStream_t of device 0 of the ctx; NULL = own */
int qo_ctx_num_devices(const qo_ctx *ctx);
void qo_ctx_destroy(qo_ctx *ctx);

/* nominal sweep (Qucs ".SP" + "S[i,j]" + "dB()" of pa-lpf-simulation.sch:59-60);
 * precision 64 or 32; every output pointer nullable; gd = -d(arg S21)/dw [s] */
int qo_sweep(qo_ctx *ctx, const qo_net *net, const double *f, int nf, int precision,
             qo_c64 *s11, qo_c64 *s21, qo_c64 *s12, qo_c64 *s22, double *gd);

typedef enum { QO_SPEC_S21_MIN_DB = 1, QO_SPEC_S21_MAX_DB = 2, QO_SPEC_S11_MAX_DB = 3, QO_SPEC_GD_MAX = 4 } qo_spec_kind;
typedef struct { int32_t kind; int32_t pad; double f_lo, f_hi, limit; } qo_spec; /* applies to grid f in [f_lo,f_hi] */
#define QO_MAX_SPEC 8

typedef enum { QO_DIST_UNIFORM = 0, QO_DIST_GAUSS3S = 1 } qo_dist;
typedef enum { QO_TOL_REL = 0, QO_TOL_ABS = 1 } qo_tol_mode;
/* one perturbed parameter: p[param] of element elem is nominal*(1+tol*x) (REL)
 * or nominal+tol*x (ABS), x in [-1,1] drawn for random variable `var`
 * (entries sharing a var share the draw, e.g. one etch delta per board) */
typedef struct { int32_t elem, param, var, mode; double tol; } qo_tol;
typedef enum { QO_MODE_REDUCE_ONLY = 0, QO_MODE_FULL_S = 1 } qo_mc_mode;

typedef struct {
    uint64_t seed, sample_offset, n_samples;
    int32_t dist, n_tol;
    const qo_tol *tol;
    int32_t mode, precision;        /* qo_mc_mode; 64 | 32 */
    int32_t hist_bins, hist_spec;   /* histogram of the worst value of spec hist_spec, in its unit */
    double hist_lo, hist_hi;
} qo_mc_cfg;

typedef struct {
    uint64_t n_pass, n_total;
    uint64_t *fail_per_spec;   /* caller array [nspec], nullable */
    uint64_t *hist;            /* caller array [hist_bins], nullable */
    double seconds;            /* device time of the kernel(s), CUDA events */
    double evals_per_s;        /* n_total * nf / seconds */
    double flops_per_eval;     /* ALG-v1 count for this network (DESIGN.md) */
} qo_mc_result;

/* Monte-Carlo yield with HOST buffers.  full_s (nullable unless mode==FULL_S):
 * planes [4][n_samples][nf] in the order S11, S21, S12, S22. */
int qo_mc_run(qo_ctx *ctx, const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec,
              const qo_mc_cfg *cfg, qo_mc_result *res, qo_c64 *full_s);

/* N-port nodal analysis on the GPU (netlist container above) */
/* spec on one S entry: kind QO_SPEC_S21_MIN_DB / QO_SPEC_S21_MAX_DB applied to |S[row][col]| (0-based) in dB */
typedef struct { int32_t kind; int32_t row, col, pad; double f_lo, f_hi, limit; } qo_nspec;
/* nominal sweep: s[nf][np][np], S[k][j] = b_k / a_j (Qucs "S[k+1,j+1]") */
int qo_nodal_sweep(qo_ctx *ctx, const qo_nodal *nd, const double *f, int nf, qo_c64 *s);
/* Monte Carlo over branch parameters (qo_tol.elem = branch index, .param = p index); counters as qo_mc_run;
 * full_s (nullable unless cfg->mode == QO_MODE_FULL_S): [n_samples][nf][np][np] */
int qo_nodal_mc_run(qo_ctx *ctx, const qo_nodal *nd, const double *f, int nf, const qo_nspec *spec, int nspec,
                    const qo_mc_cfg *cfg, qo_mc_result *res, qo_c64 *full_s);

/* The host-only part of a nodal job (needs no GPU): compile the netlist and try the static factorisation plan -- one pivot
 * order and fill pattern for the whole job, verified against a pivoted dense solve at up to 33 grid points of the nominal
 * network and at 8 vertices of the tolerance box (9 grid points each).  info[0] = plan accepted, [1] = unknowns, [2] = packed
 * non-zeros incl. fill, [3] = program length in 16-bit words; *max_multiplier (nullable) = the largest |L| entry the probes met.
 * On the device every point re-checks its own multipliers: a point above 3e6 (or NaN) sends the whole job to the kernel with
 * per-point partial pivoting, so an unprobed frequency or an interior sample cannot silently lose digits. */
int qo_nodal_analyze(const qo_nodal *nd, const double *f, int nf, const qo_mc_cfg *cfg, int info[4], double *max_multiplier);
/* Large nodal jobs (>= 4e8 points, or QO100NET_NODAL=jit) do not interpret the static plan: the library prints it as a
 * straight-line kernel for this network -- stamps, elimination and only the substitutions the observed S entries need, every
 * value a named register -- compiles it with NVRTC for sm_100a and keeps it for the life of the process.  This entry point runs
 * the same generation and compilation without a GPU (the tool the reference used, qucsator, re-factorises
 * util/pa-bias-simulation/pa-bias-simulation.sch:19-72 numerically at every point).  info[0] = compiled (0: static plan refused,
 * libnvrtc missing or a compilation error, see qo_last_error), [1] = registers per thread, [2] = stack frame bytes (0 = the whole
 * factorisation lives in registers), [3] = spill bytes, [4] = complex multiply-subtracts per point, [5] = reciprocals per point. */
int qo_nodal_jit_analyze(const qo_nodal *nd, const double *f, int nf, const qo_nspec *spec, int nspec, const qo_mc_cfg *cfg, int info[6]);

/* which factorisation the calling thread's last nodal call used: "qo_nodal_kernel<static,local>" (symbolic plan:
 * fixed pivot order and fill pattern, verified on the host against the pivoted solve; values in a thread-private array), "qo_nodal_jit_kernel"
 * (the same plan compiled into a kernel of its own, values in registers) or "qo_nodal_kernel<dense>" (per-point partial pivoting; QO100NET_NODAL=dense forces it) */
const char *qo_nodal_last_kernel(void);
/* seconds the calling thread's last nodal call spent generating + compiling its kernel (0: none needed, or taken from the process cache) */
double qo_nodal_last_compile_seconds(void);

/* The same job kept resident in HBM (tables, grid, specs uploaded once):
 *   counters layout (uint64): [0]=n_pass [1]=n_total [2..2+nspec)=fail_per_spec, then hist[hist_bins].
 * qo_plan_launch is asynchronous on the ctx stream and ADDS into counters_dev
 * (NULL = the plan's own buffer, zeroed by qo_plan_reset). full_s_dev: device
 * buffer of planes [4][n_samples][nf] for FULL_S, else NULL. */
int qo_plan_create(qo_ctx *ctx, const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec,
                   const qo_mc_cfg *cfg, qo_plan **out);
int qo_plan_num_counters(const qo_plan *plan);
int qo_plan_reset(qo_plan *plan);
int qo_plan_launch(qo_plan *plan, uint64_t sample_offset, uint64_t n_samples, uint64_t *counters_dev, qo_c64 *full_s_dev);
int qo_plan_read(qo_plan *plan, qo_mc_result *res);   /* synchronises, combines across the ctx's GPUs */
double qo_plan_flops_per_eval(const qo_plan *plan);
int qo_plan_launches(const qo_plan *plan);            /* kernels launched so far by this plan */
/* which kernel the plan launches: "qo_mc_spot_kernel" (one thread per sample: reduce-only jobs on lumped cascades with
 * <= 8 frequencies), "qo_mc_tf_kernel" (transfer-function kernel: reduce-only |S21| / |S11| / group-delay jobs on lumped
 * cascades, optionally behind one coupled-line block), "qo_mc_ladder_kernel" (straight-line ABCD-chain kernel of
 * the pcb/generic-filter ladder family), "qo_mc_lumped_kernel" (opcode interpreter) or "qo_mc_generic_kernel"
 * (microstrip).  QO100NET_KERNEL=ladder keeps jobs off the transfer-function kernel, =interp forces the interpreter.
 * "qo_mc_chain_jit_kernel": what would run on the interpreter -- a line or a measured block inside or behind the cascade
 * (util/pa-bias-simulation/pa-bias-simulation.sch:39), FULL_S behind a coupled line (util/directional-couplers/
 * dir_cpl_2.4g_20dB.trc:18-20) -- runs, from 2e10 evals per launch on (5e7 once this process or QO100NET_CACHE_DIR holds the
 * kernel; QO100NET_CHAIN=jit always, =interp never), on the interpreter's own source compiled at run time with the element
 * list, spec kinds and mode as constants (NVRTC, sm_100a): same arithmetic, no dispatch.  The name follows the last launch. */
const char *qo_plan_kernel_name(const qo_plan *plan);
/* The host-only part of that (NVRTC compiles without a GPU): fold this job's element list into the chain kernel and compile it.
 * info[0] = compiled (0: libnvrtc missing or a compilation error, see qo_last_error), [1] = registers per thread, [2] = spill
 * bytes (-1 for either when NVRTC does not echo ptxas), [3] = cubin size in bytes. */
int qo_chain_jit_analyze(const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec, const qo_mc_cfg *cfg, int info[4]);
/* what the plan decided about the transfer-function kernel.  info[0] = selected (0/1), [1] = numerator chains (2 | 4),
 * [2] = denominator form (0 none, 1 truncated |D|^2 polynomial, 2 complex D, 3 D and dD/ds for group-delay jobs), [3] = coefficient pairs kept per numerator
 * polynomial, [4] = denominator coefficients (form 1) / pairs (form 2) kept, [5] = structural degree;
 * *self_check_err = worst relative disagreement on |den|^2 between the expansion and the per-element evaluation
 * (nominal network + both ends of the tolerance box, every in-band grid point); *fused = bit mask of the specs whose
 * single-spec stretches of the grid the thread-per-sample kernel walks on one fused margin polynomial, *fused_err = the worst
 * disagreement of that margin with the unfused one, relative to |den|^2 (0 when no spec is fused).  Any output pointer may be
 * NULL.  Returns the reason string ("ok", or why the job stays on the chain kernels). */
const char *qo_plan_tf_info(const qo_plan *plan, int info[6], double *self_check_err, unsigned int *fused, double *fused_err);
/* the host-only part of qo_plan_create (network -> program, transfer-function analysis): needs no GPU.  Same outputs as
 * qo_plan_tf_info; *seconds = host time the analysis took.  An environment override qo_plan_create would refuse (an unknown
 * QO100NET_KERNEL value): info[0] = QO_ERR_ARG and the reason string says why. */
const char *qo_plan_analyze(const qo_net *net, const double *f, int nf, const qo_spec *spec, int nspec, const qo_mc_cfg *cfg,
                            int info[6], double *self_check_err, unsigned int *fused, double *fused_err, double *seconds);
/* host->device bytes qo_plan_create copied for this plan (tables, masks, program), per GPU */
uint64_t qo_plan_h2d_bytes(const qo_plan *plan);
void qo_plan_destroy(qo_plan *plan);

/* ---- reference stream: host-callable, bit-exact twins of the device code -- */
void   qo_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
double qo_variate(uint64_t seed, uint64_t sample, uint32_t var, int dist);          /* x in [-1,1] */
double qo_perturb_factor(uint64_t seed, uint64_t sample, uint32_t var, int dist, double tol);
/* the device's own stream, for the bit-exactness test: out[n_samples][n_var] = 1+tol*x */
int qo_device_perturb_factors(qo_ctx *ctx, uint64_t seed, uint64_t sample_offset, uint64_t n_samples,
                              int n_var, int dist, double tol, double *out);

/* the kernels' fast reciprocal (MUFU.RCP64H + one cubic step) applied to in[0..n), for accuracy tests */
int qo_device_rcp(qo_ctx *ctx, const double *in, size_t n, double *out);
/* the microstrip kernels' logarithm (qo_ustrip.cuh::ms_log: fdlibm reduction + degree-7 minimax, Newton reciprocal) applied to
 * in[0..n), for accuracy tests */
int qo_device_mslog(qo_ctx *ctx, const double *in, size_t n, double *out);

/* measured FP64 FMA peak of device 0 of the ctx (dependency-free DFMA loop), TFLOP/s */
int qo_measure_dfma_peak(qo_ctx *ctx, double *tflops);

const char *qo_strerror(int status);
const char *qo_last_error(void);  /* thread-local detail of the last failure ("" if none) */
const char *qo_version(void);

#ifdef __cplusplus
}
#endif
#endif
