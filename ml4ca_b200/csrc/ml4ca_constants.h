// ml4ca_constants.h -- every physical / reward / allocator constant of the ReVolt DP hot path.
//
// Plain C header (no CUDA) shared by the kernels and parsed by tests/test_constants.py, which checks
// that oracle/constants.py carries the same numbers.
//
// Provenance (reference paths relative to /root/reference):
//  * thruster geometry  lx, ly            src/qp/ROS/qp_allocator/src/qp_allocator.py:69-70
//  * thrust law F = K n|n|, K             src/qp/ROS/qp_allocator/src/qp_allocator.py:51-55,284-288
//  * force / azimuth rate limits          src/qp/ROS/qp_allocator/src/qp_allocator.py:57-58
//  * env bounds, reward coefficients      src/rl/windows_workspace/specific/customEnv.py:26,78-88,263,386-399
//  * PID saturation [69,30,80]            src/sl/SupervisedTau.py:37
//  * hull mass / damping                  NOT IN THE REFERENCE (proprietary Cybersea simulator is absent).
//                                         DECLARED STAND-IN values, calibrated so that full thrust reaches the
//                                         top speeds quoted in customEnv.py:13-18 (+1.4 m/s, 0.30 m/s, 0.52 rad/s).
#ifndef ML4CA_CONSTANTS_H_
#define ML4CA_CONSTANTS_H_

#define ML4CA_PI 3.14159265358979323846

// ---- thrusters, allocator order [port, star, bow] -----------------------------------------------------------
#define ML4CA_LX_PORT (-1.12)
#define ML4CA_LX_STAR (-1.12)
#define ML4CA_LX_BOW (1.08)
#define ML4CA_LY_PORT (-0.15)
#define ML4CA_LY_STAR (0.15)
#define ML4CA_LY_BOW (0.0)
#define ML4CA_K_STERN (0.00205)  // N / %^2
#define ML4CA_K_BOW (0.0009)     // N / %^2
#define ML4CA_FMAX_STERN (20.5)  // N
#define ML4CA_FMAX_BOW (9.0)     // N
#define ML4CA_BOW_ANGLE_FIXED (ML4CA_PI / 2.0)

// ---- SLSQP allocator (qp_allocator.py) ------------------------------------------------------------------------
#define ML4CA_QP_DF_STERN (5.0)             // max |f - f_prev| per call, N
#define ML4CA_QP_DF_BOW (2.0)
#define ML4CA_QP_DA_STERN (ML4CA_PI / 12.0)  // max |alpha - alpha_prev| per call, rad
#define ML4CA_QP_ALPHA_BOUND (2.0 * ML4CA_PI)
#define ML4CA_QP_SLACK_BOUND (1.0)
#define ML4CA_QP_W_RATE (0.25)   // Q weight of the angle-change and force-change terms
#define ML4CA_QP_CLEAN_EPS (0.01)  // |x| < eps -> 0 (qp_allocator.py:232)
#define ML4CA_BOW_THROTTLE_GAIN (2.5)  // qp_allocator.py:307 (SIMULATION == False)

// ---- stand-in hull, 3-DOF surge/sway/yaw (DECLARED, not from the reference) ---------------------------------
#define ML4CA_M11 (264.0)   // kg      (257 kg hull + surge added mass)
#define ML4CA_M22 (306.0)   // kg
#define ML4CA_M33 (322.0)   // kg m^2
#define ML4CA_XU (10.0)     // linear damping   N/(m/s)
#define ML4CA_XUU (13.8)    // quadratic        N/(m/s)^2      10*1.4 + 13.8*1.96 = 41.0 N = 2*20.5
#define ML4CA_YV (100.0)
#define ML4CA_YVV (222.0)   //                   100*0.3 + 222*0.09 = 50.0 N = 2*20.5 + 9
#define ML4CA_NR (60.0)
#define ML4CA_NRR (90.3)    //                   60*0.52 + 90.3*0.2704 = 55.6 Nm
#define ML4CA_SIM_DT (0.01) // s, one simulator sub-step (customEnv.py:79-81)
// Second DECLARED parameter set (ml4ca_env_cfg.hull_model = 1): output-error fit of the same equations to the reference's
// recorded Cybersea box tests (tools/sysid_hull.py --constrained --wrench-lag; results/all_plots/box_test/), with the
// quadratic coefficients tied to the same top speeds as above, plus a first-order lag of the thruster wrench.
#define ML4CA_H1_M11 (271.0)
#define ML4CA_H1_M22 (316.0)
#define ML4CA_H1_M33 (320.0)
#define ML4CA_H1_XU (12.3)
#define ML4CA_H1_XUU (12.13)  //                   12.3*1.4 + 12.13*1.96 = 41.0 N
#define ML4CA_H1_YV (0.0)
#define ML4CA_H1_YVV (555.6)  //                   555.6*0.09 = 50.0 N
#define ML4CA_H1_NR (106.0)
#define ML4CA_H1_NRR (1.78)   //                   106*0.52 + 1.78*0.2704 = 55.6 Nm
#define ML4CA_H1_LAG_S (0.92) // s, fitted time constant of the wrench lag (ml4ca_env_cfg.actuator_lag_s)

// ---- env (RevoltFinal, extended state, continuous angles) ---------------------------------------------------
#define ML4CA_N_SUBSTEPS 20
#define ML4CA_MAX_EP_LEN 400
#define ML4CA_BOUND_POS (8.0)
#define ML4CA_BOUND_YAW (45.0 * ML4CA_PI / 180.0)
#define ML4CA_BOUND_U (1.4)
#define ML4CA_BOUND_V (0.30)
#define ML4CA_BOUND_R (0.52)
#define ML4CA_THRUST_BOUND (100.0)
#define ML4CA_VEL_FRACTION (0.30)  // reset: velocities sampled on 0.30 * fraction (customEnv.py:145)

// ---- reward (customEnv.py:263-325) --------------------------------------------------------------------------
#define ML4CA_REW_VEL_CU (0.5)
#define ML4CA_REW_VEL_CV (0.5)
#define ML4CA_REW_VEL_CR (1.0)
#define ML4CA_REW_SIGMA_POS (1.0)   // m
#define ML4CA_REW_SIGMA_YAW (5.0)   // deg
#define ML4CA_REW_THRUST_C_BOW (0.20)
#define ML4CA_REW_THRUST_C_STERN (0.30)
#define ML4CA_REW_DTHRUST_C (0.05)
#define ML4CA_REW_DANGLE_C_BOW (0.0)
#define ML4CA_REW_DANGLE_C_STERN (0.01)

// ---- pseudoinverse + PID baseline (absent from the reference; gains are this build's own, DECLARED) ---------
#define ML4CA_PID_KP_X (30.0)
#define ML4CA_PID_KP_Y (30.0)
#define ML4CA_PID_KP_N (60.0)
#define ML4CA_PID_KD_X (90.0)
#define ML4CA_PID_KD_Y (120.0)
#define ML4CA_PID_KD_N (120.0)
#define ML4CA_PID_KI_X (1.0)
#define ML4CA_PID_KI_Y (1.0)
#define ML4CA_PID_KI_N (2.0)
#define ML4CA_PID_SAT_X (69.0)
#define ML4CA_PID_SAT_Y (30.0)
#define ML4CA_PID_SAT_N (80.0)
#define ML4CA_PID_DT (0.2)

// ---- passive nonlinear DP observer (Fossen & Strand 1999; DECLARED defaults of ml4ca_observer_cfg_default) -----
// Per DOF: K11 = -2 (zeta_n - lambda) w_c / w_o, K12 = 2 w_o (zeta_n - lambda), K2 = w_c = CUTOFF_RATIO w_o,
// K4 = K4_PER_MASS diag(m11, m22, m33) of the selected hull, K3 = K3_PER_K4 K4; 1/T_b <= K3/K4 < w_o < w_c.
// Mirrored in tests/observer_oracle.py and checked there by tests/test_observer_cpu.py.
#define ML4CA_OBS_NOTCH_DAMPING (1.0)   // zeta_n
#define ML4CA_OBS_WAVE_DAMPING (0.1)    // lambda
#define ML4CA_OBS_CUTOFF_RATIO (1.2)    // w_c / w_o
#define ML4CA_OBS_BIAS_TIME_S (0.0)     // T_b, 0 = infinity
#define ML4CA_OBS_K4_PER_MASS (0.2)     // 1/s^2
#define ML4CA_OBS_K3_PER_K4 (0.2)       // 1/s
#define ML4CA_OBS_PEAK_FREQUENCY (1.5)  // rad/s: the fixed w_o a DPObserver starts with
#define ML4CA_OBS_OMEGA_MIN (0.1)       // rad/s: the kernel clamps every w_o (NaN included) into [MIN, MAX]
#define ML4CA_OBS_OMEGA_MAX (10.0)
#define ML4CA_OBS_STATE_ROWS 15         // xi1[3], xi2[3], eta[3], nu[3], b[3]

// ---- DP reference model (Fossen 2011 section 12.1; DECLARED defaults of ml4ca_refmodel_cfg_default) --------------
// Per DOF (N, E, psi): eta_d / r = w^3 / ((s + w)(s^2 + 2 zeta w s + w^2)) with |v_d| <= V_MAX, |a_d| <= A_MAX.  Tuned
// on the float64 closed loop of PID + feed-forward + pseudoinverse over the box test (DESIGN.md section 4).
// Mirrored in tests/refmodel_oracle.py and checked there by tests/test_refmodel_cpu.py.
#define ML4CA_REF_ZETA_N (1.0)
#define ML4CA_REF_ZETA_E (1.0)
#define ML4CA_REF_ZETA_PSI (1.0)
#define ML4CA_REF_OMEGA_N (0.2)      // rad/s
#define ML4CA_REF_OMEGA_E (0.2)
#define ML4CA_REF_OMEGA_PSI (0.25)
#define ML4CA_REF_V_MAX_N (0.15)     // m/s
#define ML4CA_REF_V_MAX_E (0.1)      // m/s
#define ML4CA_REF_V_MAX_PSI (0.1)    // rad/s
#define ML4CA_REF_A_MAX_N (0.05)     // m/s^2
#define ML4CA_REF_A_MAX_E (0.02)     // m/s^2
#define ML4CA_REF_A_MAX_PSI (0.02)   // rad/s^2
#define ML4CA_REF_STATE_ROWS 9       // eta_d[3], v_d[3], a_d[3]

#endif  // ML4CA_CONSTANTS_H_
