// Fused MaxEnt alpha sweep for sm_100a (B200), "spectrum per CTA".
//
// One CTA of 8 warps owns one spectrum at a time (persistent CTAs, atomic work counter, as many CTAs per SM as
// registers and shared memory allow: two) and runs the whole alpha mesh for it.
// Round 2 measured the alternatives on B200 (profiles/r02_ab_*.log): four 4-warp CTAs per SM are 10 % slower, three
// 4-warp CTAs at 168 registers 3 % slower than two 8-warp CTAs -- the FP64 pipe is 62-68 % busy in all three, so the
// idle third is not a matter of how the warps are grouped.  The Levenberg-Marquardt iteration of the reference
// (levenberg_minimizer.py:123-248) asks for Q(v - dv(mu)) at a chain of damping values
// mu, 1.3 mu, 1.3^2 mu ... that is decided by comparisons of the Q values.  Instead of evaluating the
// chain one trial at a time (latency bound), the CTA *speculates*: it plans the next up-to-8 damping
// values the reference would visit, factorises the 8 shifted Hessians (one warp per matrix, DMMA-blocked "lean"
// L D L^T) and evaluates the 8 trial vectors in ONE pass over
// V' where the 8 trials are the M dimension of the FP64 tensor-core MMA (m8n8k4):
//     T-pass:  x = V' t_b ; H = D exp(x) ; y_b = V'^T H ; S_b ; w_b -> scratch      (8 trials)
//     H-pass:  Z = V'^T diag(w) V'                                                   (accepted point)
// The reference's state machine is then replayed on the tabulated Q values, so the sequence of accepted
// steps, the damping schedule and all comparisons are exactly those of the reference; speculation only
// changes WHEN a value is computed.  Every point is evaluated once: the accepted trial's chi2, S, y and
// w = dH/dx are reused for the next gradient / Hessian (the reference recomputes them), and Z is reused
// when alpha changes (Z does not depend on alpha).
//
// All small dense algebra works on 8x8 tiles in the accumulator ("C") layout of the MMA: lane L
// (r = L/4, q = L%4) holds T[r][2q], T[r][2q+1].  With the k index of the MMA permuted (k-step e uses
// columns 2q+e) two C-layout tiles multiply as X Y^T straight from their registers (mma_nt), which
// gives the Cholesky trailing updates, J = eta Z Lambda Z + alpha Z and f = Z u without any layout
// conversion.  tools/lane_model.py is the numpy model these routines were derived from.
//
// V' streams L2 -> shared memory with 1-D TMA bulk copies (cp.async.bulk + mbarrier) in the
// swizzled 8x8-tile layout written by mx_layout_V.  A bulk copy costs the CTA ~360 cycles whatever its size
// (tools/tma_stream_bench.cu), so a chunk is one copy of NWARP k-tiles: one tile per warp and step in the T-pass.
//
// Instantiations: NT = 4..10 tiles of 8 singular-space columns (n_sv <= 80) keep every matrix in shared memory and
// registers as described; NT = 12, 16, 24, 32 (n_sv <= 256, "wide") run the same code with Z, J and the factors in a
// per-CTA slice of the global workspace and V' read from L2 directly (see is_wide below).
#pragma once
#include <stdlib.h>
#include "mx_common.cuh"

namespace mx2 {

using mx::SweepArgs;
using mx::dmma;
using mx::tile_off;

constexpr int NWARP = 8;        // the fixed-order reduction trees over the warps are written for 8
constexpr int CTAS_PER_SM = 2;  // CTAs per SM the kernel is compiled for: register cap = 64K / (CTAs x threads)
constexpr int NTHR = NWARP * 32;
constexpr int NKG = NWARP / 2;  // k-groups of the H-pass (two warps -- the two halves of the triangle -- per group)
constexpr int CH = NWARP;       // k-tiles (8 omega rows each) per staged chunk = one per warp in the T-pass, two per k-group in the H-pass
constexpr int MAXB = 8;        // unique trials per batch = M of the MMA
constexpr int NTAB = 32;       // damping values tabulated per batch (several may share one unique trial)
constexpr int NROWS = 9;       // scratch rows per CTA: 8 trials + 1 carried candidate
constexpr int ID_NONE = -1, ID_CARRY = 8;

// ------------------------------------------------------------------------------------------
// PTX helpers: mbarrier + TMA bulk copy
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t* b, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(b)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(b)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// L2 policy for the per-CTA scratch rows (w = dH/dx of the evaluated trials): they are rewritten every batch and read
// back by the H-pass, so they should stay in L2 while the A(alpha) output streams through (written once, never read)
__device__ __forceinline__ uint64_t l2_evict_last_policy() {
    uint64_t pol;
    asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void st_keep_v2(double* p, double x, double y, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1, %2}, %3;" ::"l"(p), "d"(x), "d"(y), "l"(pol) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

__device__ __forceinline__ double shfl(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }
__device__ __forceinline__ double shfl_xor(double v, int m) { return __shfl_xor_sync(0xffffffffu, v, m); }
__device__ __forceinline__ double quadreduce(double x) { x += shfl_xor(x, 1); x += shfl_xor(x, 2); return x; }
__device__ __forceinline__ double colreduce(double x) { x += shfl_xor(x, 4); x += shfl_xor(x, 8); x += shfl_xor(x, 16); return x; }
__device__ __forceinline__ double warp_sum(double x) { return colreduce(quadreduce(x)); }
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// 1/sqrt(a) for a > 0: MUFU.RSQ64H seed (about 2^-20) + two Newton steps (quadratic: 2^-40, then rounding level);
// shorter dependent chain than the library rsqrt(), which sits on the critical path of the Cholesky panel
__device__ __forceinline__ double rsqrt_nr(double a) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    double h = 0.5 * y;
    double e = fma(-a * y, y, 1.0);
    y = fma(h, e, y);
    h = 0.5 * y;
    e = fma(-a * y, y, 1.0);
    return fma(h, e, y);
}

// 1/a: MUFU.RCP64H seed + two Newton steps
__device__ __forceinline__ double rcp_nr(double a) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    double e = fma(-a, y, 1.0);
    y = fma(y, e, y);
    e = fma(-a, y, 1.0);
    return fma(y, e, y);
}

// c += X Y^T for two 8x8 tiles in C layout (k permuted: k-step e uses columns 2q+e)
__device__ __forceinline__ void mma_nt(double (&c)[2], double x0, double x1, double y0, double y1) {
    dmma(c, x0, y0);
    dmma(c, x1, y1);
}

__host__ __device__ constexpr int tri(int I, int J) { return I * (I + 1) / 2 + J; }

// ------------------------------------------------------------------------------------------
// sizes of the "lean" blocked Cholesky (see below): how many tiles of the factor a warp parks in shared memory
// ------------------------------------------------------------------------------------------
constexpr int LEAN_RTILES = 10;    // strictly-lower tiles of the factor a warp keeps in registers
__host__ __device__ constexpr int lean_nsm(int NT) {
    int nsm = 0;
    while (nsm < NT && (NT - 1 - nsm) * (NT - nsm) / 2 > LEAN_RTILES) ++nsm;
    return nsm;
}
__host__ __device__ constexpr int lean_nsmt(int NT) {          // strictly-lower tiles of the factor a warp parks in shared memory
    const int nsm = lean_nsm(NT);
    return NT * (NT - 1) / 2 - (NT - 1 - nsm) * (NT - nsm) / 2;
}
template <int NT>
struct Lean {
    static constexpr int NSM = lean_nsm(NT);                                   // block columns kept in shared memory
    static constexpr int NREG = (NT - 1 - NSM) * (NT - NSM) / 2;               // strictly-lower tiles kept in registers
    static constexpr int NSMT = NT * (NT - 1) / 2 - NREG;                      // tiles per warp in shared memory
    static constexpr int RDIM = NREG > 0 ? NREG : 1;
    __host__ __device__ static constexpr int before(int J, int from) {
        int o = 0;
        for (int j = from; j < J; ++j) o += NT - 1 - j;
        return o;
    }
    __host__ __device__ static constexpr int sidx(int I, int J) { return before(J, 0) + I - J - 1; }
    __host__ __device__ static constexpr int ridx(int I, int J) { return J >= NSM ? before(J, NSM) + I - J - 1 : 0; }
};

// Staging buffers of the V' stream: at least two (one being consumed, one in flight), and enough area for what the
// ring is reused for between passes: Zfull (NT x NT tiles), the parked Cholesky tiles of every solving warp, the
// per-warp y partials of the T-pass.
// warps that factorise at the same time: all of them up to 7 tiles; beyond that every warp parks so many tiles that
// a full house would cost the second CTA per SM, so half the warps solve in twice the rounds
__host__ __device__ constexpr int solver_warps(int NT) { return NT <= 7 ? NWARP : NWARP / 2; }
__host__ __device__ constexpr int stage_count(int NT) {
    int need = NT * NT;                                                          // in 8x8 tiles
    if (solver_warps(NT) * lean_nsmt(NT) > need) need = solver_warps(NT) * lean_nsmt(NT);
    if (NWARP * NT > need) need = NWARP * NT;
    // partial Z tiles of the H-pass: Zfull + (NKG - 1) triangles, minus what J and the trial vectors behind the ring hold
    const int hneed = NT * NT + (NKG - 2) * (NT * (NT + 1) / 2) - 2 * NT;
    if (hneed > need) need = hneed;
    int nst = (need + CH * NT - 1) / (CH * NT);
    if (nst < 2) nst = 2;
    return nst;
}

// ------------------------------------------------------------------------------------------
// shared-memory layout (offsets in doubles)
// ------------------------------------------------------------------------------------------
// Wide singular spaces (NT > 10 tiles, n_sv up to 256): Z, J and the factors of the trial systems do not fit in shared
// memory any more.  They live in a per-CTA slice of the global workspace (L2-resident), V' is read straight from L2
// (no staging ring), one CTA per SM with the full register file; everything else -- the replay of the damping search,
// the pointwise map, the order of every sum inside a spectrum -- is the code of the narrow instantiations.
__host__ __device__ constexpr bool is_wide(int NT) { return NT > 10; }
__host__ __device__ constexpr long long wide_doubles(int NT) {     // Zfull + J + one factor per warp (diagonal slots = U tiles)
    return is_wide(NT) ? (long long)(NT * NT + (1 + NWARP) * (NT * (NT + 1) / 2)) * 64 : 0;
}

template <int NT>
struct Lay {
    static constexpr bool WIDE = is_wide(NT);
    static constexpr int SP = 8 * NT;
    static constexpr int NTRI = NT * (NT + 1) / 2;
    static constexpr int STAGE_D = CH * NT * 64;
    static constexpr int NST = WIDE ? 0 : stage_count(NT);
    static constexpr int LEAN_AREA = WIDE ? 0 : solver_warps(NT) * Lean<NT>::NSMT * 64;
    static constexpr int STAGE_AREA = WIDE ? NWARP * 8 * SP                     // wide: only the y partials of the T-pass
                                           : (NST * STAGE_D > LEAN_AREA ? NST * STAGE_D : LEAN_AREA);
    static constexpr int o_stage = 0;                              // NST x STAGE_D ; aliases: Zfull [NT*NT*64], yred [NWARP][8][SP], parked Cholesky tiles
    static constexpr int o_J = o_stage + STAGE_AREA;            // NTRI tiles, C layout (also: partial Z tiles of the H-pass, parked tiles of the log-det)
    static constexpr int o_tb = o_J + (WIDE ? 0 : NTRI * 64);      // [8][SP] trial vectors t_b = v - dv_b  (the accepted one IS the new v, levenberg_minimizer.py:239)
    static constexpr int o_yb = o_tb + MAXB * SP;                  // [8][SP]
    static constexpr int o_ctb = o_yb + MAXB * SP;                 // carried candidate: t, y
    static constexpr int o_cy = o_ctb + SP;
    static constexpr int o_v = o_cy + SP;
    static constexpr int o_f = o_v + SP;
    static constexpr int o_rhs = o_f + SP;
    static constexpr int o_u = o_rhs + SP;
    static constexpr int o_gt = o_u + SP;
    static constexpr int o_xi = o_gt + SP;
    static constexpr int o_lam = o_xi + SP;
    static constexpr int o_ycur = o_lam + SP;
    static constexpr int o_jd = o_ycur + SP;                       // diagonal of J
    static constexpr int o_sred = o_jd + SP;                       // [NWARP][8] entropy partials
    static constexpr int o_ctl = o_sred + NWARP * 8;                      // Ctl block (192 doubles reserved)
    static constexpr int o_bar = o_ctl + 192;                      // 2*NST mbarriers
    static constexpr int total = o_bar + 2 * NST;
    static_assert(WIDE || NT * NT * 64 <= NST * STAGE_D, "Zfull must fit in the staging area");
    static_assert(NWARP * 8 * SP <= STAGE_AREA, "yred must fit in the staging area");
    static_assert(WIDE || solver_warps(NT) * Lean<NT>::NSMT * 64 <= STAGE_AREA, "the parked tiles of the solver warps must fit in the staging area");
    static_assert(WIDE || Lean<NT>::NSMT <= NTRI, "the parked tiles of the log-det factorisation must fit in the J area");
    static_assert(WIDE || NT * NT * 64 + (NKG - 1) * NTRI * 64 <= o_ctb, "partial Z tiles of the H-pass must fit behind Zfull");
};

enum { PH_FIRST = 0, PH_PUMP, PH_PROBE, PH_WALK, PH_DONE };

struct LM {
    int phase, dv, dvnew;
    double mu, Q0, Q1, Q2, nuf;
};

// control block, lives in shared memory; written by thread 0 (and warp 0), read by all after a barrier
struct Ctl {
    LM lm;
    double alpha, c0, chi2_cur, S_cur, Q1cur;
    double bmu[NTAB];          // damping of every table entry of the current batch
    double umu[NROWS];         // damping of the unique trials (index 8 = carried candidate)
    double uQ[NROWS], uchi2[NROWS], uS[NROWS];   // per unique trial (index 8 = carried candidate)
    double pq[MAXB];           // planning: pretended Q of the planned unique trials
    double maxf;
    int bslot[NTAB];           // table entry -> unique trial
    int urow[NROWS];           // scratch row of each unique trial (8 = carried)
    int ufail[NROWS];
    int nb, nuniq;
    double jdmin;              // smallest |J_kk| (quick test for equivalent dampings)
    int spec, ia, it, nq, ns, dir_up, cur_row, action, conv, last_len, ns_it0, ntrial, nbatch;
    unsigned gchunk;           // chunks streamed so far (pipeline phase bookkeeping)
    long long t_last;          // phase timers (clock64 of thread 0), see MX_PHASE_*
    long long tph[8];
#ifdef MX_TPROF
    long long pf[16];
#endif
};
enum { PHT_PLAN = 0, PHT_SOLVE, PHT_TPASS, PHT_HPASS, PHT_GRAD, PHT_FORMJ, PHT_OTHER, PHT_REPLAY };
static_assert(sizeof(Ctl) <= 192 * sizeof(double), "Ctl must fit its reserved block");

// Levenberg-Marquardt damping search of one iteration, levenberg_minimizer.py:190-233, as a resumable
// machine: `look(mu, kind, Qref, Q, id)` returns false when Q(v - dv(mu)) is not tabulated yet.
template <class Look>
__device__ bool lm_run(LM& s, double nu, double max_mu, double eps_nu, Look&& look) {
    for (;;) {
        switch (s.phase) {
            case PH_FIRST: {                                   // dv = solve(J + mu) ; Q1 = Q(v - dv)      (:192-199)
                double Q; int id;
                if (!look(s.mu, 0, s.Q0, Q, id)) return false;
                s.Q1 = Q; s.dv = id; s.phase = PH_PUMP;
                break;
            }
            case PH_PUMP: {                                    // while (Q1 > Q0 or isnan(Q1)) and mu < max_mu   (:203-206)
                if ((s.Q1 > s.Q0 || isnan(s.Q1)) && s.mu < max_mu) {
                    const double m2 = s.mu * nu;
                    double Q; int id;
                    if (!look(m2, 0, s.Q0, Q, id)) return false;
                    s.mu = m2; s.Q1 = Q; s.dv = id;
                    break;
                }
                s.phase = PH_PROBE;
                break;
            }
            case PH_PROBE: {                                   // dv2 = solve(J + nu*mu) ; Q2              (:209-224)
                double Q; int id;
                if (!look(nu * s.mu, 1, s.Q1, Q, id)) return false;
                s.Q2 = Q;
                if (s.Q2 < s.Q1) { s.nuf = nu; s.mu *= nu; s.Q2 = s.Q1; s.dvnew = id; }
                else { s.nuf = 1.0 / nu; s.mu /= s.nuf; s.dvnew = s.dv; }
                s.Q1 = INFINITY;
                s.phase = PH_WALK;
                break;
            }
            case PH_WALK: {                                    // while Q2 < Q1 and mu < max_mu and mu > nu*eps (:226-233)
                if (s.Q2 < s.Q1 && s.mu < max_mu && s.mu > eps_nu) {
                    const double m2 = s.mu * s.nuf;
                    double Q; int id;
                    if (!look(m2, 2, s.Q2, Q, id)) return false;
                    s.Q1 = s.Q2; s.dv = s.dvnew; s.mu = m2; s.dvnew = id; s.Q2 = Q;
                    break;
                }
                s.phase = PH_DONE;
                return true;
            }
            default: return true;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Replay of the damping search on the tabulated trials and, when a value is missing, the plan of the next batch.
// Run by ONE warp (all 32 lanes, warp-uniform); everything it decides goes through the control block.
// jdv = diagonal of J, tb / yb = trial vectors and their y of the last batch ([8][SP]), ctb / cy = the carried candidate.
// Sets ctl.conv = 1 when the iteration's search is decided, otherwise ctl.nuniq / umu / bmu describe the next batch.
// ------------------------------------------------------------------------------------------
template <bool MARQ, class Tick>
__device__ __forceinline__ void replay_and_plan(Ctl& ctl, const SweepArgs& a, double eps_nu, int s, int SP, int lane,
                                                const double* __restrict__ jdv, const double* __restrict__ tb,
                                                const double* __restrict__ yb, double* __restrict__ ctb,
                                                double* __restrict__ cy, bool timing, Tick&& tick) {
    (void)timing;
    auto shift_of = [&](int i, double mu) -> double { return MARQ ? mu * jdv[i] : mu; };
    // The whole warp runs the (scalar, warp-uniform) state machine.  The tables live in registers:
    // lane i holds table entry i (damping, unique trial) and unique trial i (damping, Q, failed);
    // searches are ballots, reads are shuffles.
    LM L = ctl.lm;
    int ns = ctl.ns, nq = ctl.nq;
    
    const double jdmin = ctl.jdmin;
    const int nb0 = ctl.nb, nu0 = ctl.nuniq;
    int carry_row = ctl.urow[ID_CARRY];
    double t_mu = lane < nb0 ? ctl.bmu[lane] : 0.0;
    int t_slot = lane < nb0 ? ctl.bslot[lane] : 0;
    const bool uvalid = lane < nu0 || (lane == ID_CARRY && carry_row >= 0);
    double u_mu = uvalid ? ctl.umu[lane] : 0.0;
    double u_Q = uvalid ? ctl.uQ[lane] : 0.0;
    int u_fail = uvalid ? ctl.ufail[lane] : 0;
    __syncwarp();         // every lane has its copy of the control block before any lane updates it below
    // two dampings are equivalent when they give bitwise the same matrix J + shift(mu).  The entry
    // with the smallest |J_kk| can only round to the same value if they differ by less than two of
    // its ulps: cheap per-lane pre-test, the full comparison is rarely reached
    auto maybe = [&](double ma, double mb) -> bool {
        return ma == mb || !(fabs(ma - mb) > 4.5e-16 * (jdmin + fmax(ma, mb)));
    };
    auto equiv_full = [&](double ma, double mb) -> bool {
        if (ma == mb) return true;
        bool same = true;
        for (int k = lane; k < s; k += 32) {
            const double jd = jdv[k];
            same = same && ((jd + shift_of(k, ma)) == (jd + shift_of(k, mb)));
        }
        return __all_sync(0xffffffffu, same);
    };
    auto look_real = [&](double mu, int, double, double& Q, int& id) -> bool {
        const unsigned m = __ballot_sync(0xffffffffu, lane < nb0 && t_mu == mu);
        id = -1;
        if (m) id = __shfl_sync(0xffffffffu, t_slot, __ffs(m) - 1);
        else {
            const bool have_c = carry_row >= 0;
            unsigned cm = __ballot_sync(0xffffffffu, (lane < nu0 || (lane == ID_CARRY && have_c)) && maybe(mu, u_mu));
            while (cm && id < 0) {
                const int u = __ffs(cm) - 1;
                cm &= cm - 1;
                if (equiv_full(mu, shfl(u_mu, u))) id = u;
            }
        }
        if (id < 0) return false;
        Q = shfl(u_Q, id);
        ++ns; if (!__shfl_sync(0xffffffffu, u_fail, id)) ++nq;
        return true;
    };
    const int done = lm_run(L, a.nu, a.max_mu, eps_nu, look_real) ? 1 : 0;
    tick(PHT_REPLAY);
    if (!done) {
        // carry the live candidate of the old batch (its dv, y, chi2, S, damping and scratch row)
        const int live = (L.phase == PH_WALK) ? L.dvnew : (L.phase == PH_PROBE ? L.dv : ID_NONE);
        if (live >= 0 && live < MAXB) {
            for (int i = lane; i < SP; i += 32) {
                ctb[i] = tb[live * SP + i];
                cy[i] = yb[live * SP + i];
            }
            const double lmu = shfl(u_mu, live), lQ = shfl(u_Q, live);
            const int lfail = __shfl_sync(0xffffffffu, u_fail, live);
            carry_row = ctl.urow[live];
            if (lane == ID_CARRY) {
                u_mu = lmu; u_Q = lQ; u_fail = lfail;
                ctl.uQ[ID_CARRY] = lQ; ctl.uchi2[ID_CARRY] = ctl.uchi2[live]; ctl.uS[ID_CARRY] = ctl.uS[live];
                ctl.ufail[ID_CARRY] = lfail; ctl.urow[ID_CARRY] = carry_row; ctl.umu[ID_CARRY] = lmu;
            }
            if (L.phase == PH_WALK) L.dvnew = ID_CARRY; else L.dv = ID_CARRY;
        } else if (live == ID_NONE) {
            carry_row = -1;
            if (lane == 0) ctl.urow[ID_CARRY] = -1;
        }
        __syncwarp();
        // plan: continue copies of the machine with pretended outcomes to list the next dampings.
        // While the direction of this iteration's walk is not known yet (no probe outcome), BOTH
        // branches are planned: the downward walk gets most of the budget (78 % of the iterations of
        // the benchmark spectra walk down, 98 % of those that follow an upward one; tools/lm_trace.py),
        // the upward walk the rest.  A pump (Q rises: mu *= nu until it does not) continues on the
        // upward grid, so it is planned upward at full width.
        int np = 0, npu = 0;
        int budget = MAXB;
        bool dir = true;
        const bool undecided = (L.phase == PH_FIRST || L.phase == PH_PROBE);
        if (undecided) { dir = false; budget = ctl.dir_up ? MAXB - 1 : MAXB - 2; }
        else if (L.phase == PH_WALK) dir = (L.nuf == a.nu);
        LM P = L;
        const bool have_carry = carry_row >= 0;
        const double cmu = shfl(u_mu, ID_CARRY), cQ = shfl(u_Q, ID_CARRY);
        double p_mu = 0.0, pu_mu = 0.0, pu_q = 0.0;       // planned table entry / unique trial of this lane
        int p_slot = 0;
        auto find_or_add = [&](double mu, int kind, double Qref, double& Q, int& id) -> bool {
            if (have_carry && maybe(mu, cmu) && equiv_full(mu, cmu)) { Q = cQ; id = ID_CARRY; return true; }
            const unsigned m = __ballot_sync(0xffffffffu, lane < np && p_mu == mu);
            if (m) {
                const int u = __shfl_sync(0xffffffffu, p_slot, __ffs(m) - 1);
                Q = shfl(pu_q, u); id = 100 + u;
                return true;
            }
            unsigned cm = __ballot_sync(0xffffffffu, lane < npu && maybe(mu, pu_mu));
            while (cm) {
                const int u = __ffs(cm) - 1;
                cm &= cm - 1;
                if (equiv_full(mu, shfl(pu_mu, u))) {
                    if (np < NTAB) { if (lane == np) { p_mu = mu; p_slot = u; } ++np; }
                    Q = shfl(pu_q, u); id = 100 + u;
                    return true;
                }
            }
            if (npu >= budget || np == NTAB) return false;
            double pv;
            if (kind == 0) pv = isnan(Qref) ? 0.0 : Qref;                        // first trial / pump: "accepted"
            else pv = Qref - (1.0 + fabs(Qref));                                  // walk: "still improving"
            if (lane == np) { p_mu = mu; p_slot = npu; }
            if (lane == npu) { pu_mu = mu; pu_q = pv; }
            id = 100 + npu; Q = pv; ++np; ++npu;
            return true;
        };
        auto look_plan = [&](double mu, int kind, double Qref, double& Q, int& id) -> bool {
            if (!find_or_add(mu, kind, Qref, Q, id)) return false;
            if (kind == 1) {
                // the probe decides the direction: steer this run; a probe that IS the current candidate
                // (bitwise the same shifted matrix) gives Q2 == Q1, i.e. "not lower"
                if (id == P.dv) Q = Qref;
                else Q = dir ? Qref - (1.0 + fabs(Qref)) : Qref + (1.0 + fabs(Qref));
            }
            return true;
        };
        // Fast paths for the three common situations: the dampings the machine would visit are written
        // down directly, with the machine's own arithmetic (mu * nu, mu / (1/nu), mu * (1/nu), ...), instead
        // of running it on pretended outcomes.  The plan is only a proposal -- the replay above decides
        // everything on real values and re-plans when an entry is missing -- so a fast path can cost
        // speculation efficiency but never change a result.
        bool fast = false;
        {
            const double nu = a.nu, inu = 1.0 / a.nu;
            auto add_unique = [&](double mu) {
                if (lane == np) { p_mu = mu; p_slot = npu; }
                if (lane == npu) { pu_mu = mu; pu_q = 0.0; }
                ++np; ++npu;
            };
            if (L.phase == PH_PUMP && !have_carry && !maybe(L.mu * nu, L.mu)) {
                double m = L.mu;                       // pump: mu *= nu until Q stops rising (:203-206)
                for (int k = 0; k < MAXB; ++k) { m = m * nu; add_unique(m); }
                fast = true;
            } else if (L.phase == PH_WALK && have_carry && cmu == L.mu && !maybe(L.mu * L.nuf, L.mu)) {
                double m = L.mu;                       // walk: mu *= nuf while Q improves (:226-233)
                for (int k = 0; k < MAXB; ++k) { m = m * L.nuf; add_unique(m); }
                fast = true;
            } else if (L.phase == PH_FIRST && !have_carry && L.mu > 64.0 * eps_nu && L.mu < a.max_mu / 64.0 &&
                       !maybe(L.mu * nu, L.mu)) {
                const double m0 = L.mu, m1 = nu * m0;
                add_unique(m0);                        // dv = solve(J + mu)            (:192)
                add_unique(m1);                        // dv2 = solve(J + nu * mu)      (:209)
                const int ndown = ctl.dir_up ? MAXB - 3 : MAXB - 4;
                double m = m0 / inu;                   // probe lost: mu /= nuf, nuf = 1/nu   (:221-224)
                for (int k = 0; k <= ndown; ++k) {
                    m = m * inu;
                    if (k == 0) {                      // first walk point = mu again, up to rounding
                        if (m == m0) continue;
                        if (equiv_full(m, m0)) { if (lane == np) { p_mu = m; p_slot = 0; } ++np; continue; }
                    }
                    if (npu < MAXB) add_unique(m);
                }
                m = m0 * nu;                           // probe won: mu *= nu, walk upward   (:214-218)
                while (npu < MAXB) { m = m * nu; add_unique(m); }
                fast = true;
            }
        }
        if (!fast) {
            lm_run(P, a.nu, a.max_mu, eps_nu, look_plan);
            if (undecided && npu < MAXB) {         // the other branch with what is left of the batch
                P = L;
                dir = true;
                budget = MAXB;
                lm_run(P, a.nu, a.max_mu, eps_nu, look_plan);
            }
        }
        if (lane < np) { ctl.bmu[lane] = p_mu; ctl.bslot[lane] = p_slot; }
        if (lane < npu) {
            ctl.umu[lane] = pu_mu;
            ctl.urow[lane] = (carry_row >= 0 && lane >= carry_row) ? lane + 1 : lane;   // skip the carried row
            ctl.ufail[lane] = 0;
        }
        if (lane == 0) { ctl.nb = np; ctl.nuniq = npu; ctl.ntrial += npu; ctl.nbatch += 1; }
#ifdef MX_PLANPROF
        // diagnostics: charge the planning time to slot 0 (fast paths) or 6 (generic planner); slot 4
        // counts generic plans, slot 5 fast plans
        if (timing && lane == 0) {
            const long long t = clock64();
            ctl.tph[fast ? 0 : 6] += t - ctl.t_last; ctl.t_last = t;
            ctl.ntrial -= npu;                  // n_trial output = number of generic plans, by phase
            ctl.ntrial += fast ? 0 : (L.phase == PH_FIRST ? 1 : L.phase == PH_PUMP ? 1000 : L.phase == PH_PROBE ? 1000000 : 100000000);
        }
#endif
    }
    if (lane == 0) { ctl.lm = L; ctl.ns = ns; ctl.nq = nq; ctl.conv = done; }
}

// ------------------------------------------------------------------------------------------
// "lean" blocked L D L^T factorisation of a shifted Hessian by ONE warp: left-looking, at most 10 strictly-lower tiles
// stay in registers, the leading block columns are parked in a per-warp slice of shared memory, the diagonal tiles are
// dropped once the inverse U = L_d^{-T} of their unit factor is known.  ~100 registers per thread, so every warp of the
// CTA factorises its own matrix at the same time.  The stored tiles are Y = L D (unscaled columns) and the reciprocal
// pivots 1/d; a Cholesky factor would need 1/sqrt(d) per pivot as well -- a fifth of the solver's instructions on B200
// (profiles/r02a_sweep2_stalls_by_line.txt) for no numerical benefit.  A non-positive pivot = not positive definite.
// ------------------------------------------------------------------------------------------
// strictly-lower tile (I, J) of the factor: shared memory for the leading columns, registers for the rest
template <int NT>
__device__ __forceinline__ double2 lean_tile(const double* __restrict__ Lsm, const double (&R)[Lean<NT>::RDIM][2], int I, int J,
                                             int lane) {
    if (J < Lean<NT>::NSM) return *reinterpret_cast<const double2*>(Lsm + Lean<NT>::sidx(I, J) * 64 + 2 * lane);
    return make_double2(R[Lean<NT>::ridx(I, J)][0], R[Lean<NT>::ridx(I, J)][1]);
}

// block column JB: C[I] = in(I, JB) - sum_{K<JB} L[I][K] L[JB][K]^T, Cholesky of the diagonal tile together with an
// identity tile (-> U = L_d^{-T}), L[I][JB] = C[I] U for the tiles below (same arithmetic as chol_panel above)
// With FWD the forward substitution z = L^{-1} rhs rides along: block jb of z is formed as soon as block column jb of
// the factor is final, so its dependent chain (dot products, two shuffle reductions) overlaps the pivot chain of the
// next block column instead of following the factorisation (same arithmetic as a separate forward sweep).
template <int NT, int JB, bool FWD, class Load>
__device__ __forceinline__ void lean_steps(Load& load, double* __restrict__ Lsm, double (&R)[Lean<NT>::RDIM][2], double (&U)[NT][2],
                                           bool& ok, double& logdet, bool want_logdet, int r, int q, int lane,
                                           const double* __restrict__ rhs, double* __restrict__ zscr, double* __restrict__ dinv) {
    if constexpr (JB < NT) {
        constexpr int NC = NT - JB;
        double C[NC][2];
#pragma unroll
        for (int i = 0; i < NC; ++i) { const double2 t = load(JB + i, JB); C[i][0] = t.x; C[i][1] = t.y; }
#pragma unroll
        for (int K = 0; K < JB; ++K) {
            // stored tiles are Y = L D (unscaled columns); the update is Y_i D^-1 Y_JB^T
            const double2 y = lean_tile<NT>(Lsm, R, JB, K, lane);
            const double2 dk = *reinterpret_cast<const double2*>(dinv + 8 * K + 2 * q);
            const double ys0 = y.x * dk.x, ys1 = y.y * dk.y;
            mma_nt(C[0], -y.x, -y.y, ys0, ys1);
#pragma unroll
            for (int i = 1; i < NC; ++i) {
                const double2 x = lean_tile<NT>(Lsm, R, JB + i, K, lane);
                mma_nt(C[i], -x.x, -x.y, ys0, ys1);
            }
        }
        double E[2];
        E[0] = (r == 2 * q) ? 1.0 : 0.0;
        E[1] = (r == 2 * q + 1) ? 1.0 : 0.0;
        double(&P0)[2] = C[0];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int jq = j >> 1, je = j & 1;
            const double ajj = shfl(P0[je], 4 * j + jq);
            const double lk0 = shfl(P0[je], 8 * q + jq);              // a[2q][j]
            const double lk1 = shfl(P0[je], 8 * q + 4 + jq);          // a[2q+1][j]
            const int src = (lane & ~3) | jq;
            const double lp = shfl(P0[je], src);                      // a[r][j]
            const double le = shfl(E[je], src);
            if (!(ajj > 0.0)) ok = false;
            if (want_logdet) logdet += log(ajj);
            const double inv = rcp_nr(ajj);
            const double p0 = lp * lk0, p1 = lp * lk1, e0 = le * lk0, e1 = le * lk1;
            if (2 * q > j) { P0[0] = fma(-p0, inv, P0[0]); E[0] = fma(-e0, inv, E[0]); }
            if (2 * q + 1 > j) { P0[1] = fma(-p1, inv, P0[1]); E[1] = fma(-e1, inv, E[1]); }
            if (lane == 0) dinv[8 * JB + j] = inv;                   // 1 / d_j, kept in this warp's row of shared memory
        }
        __syncwarp();
        U[JB][0] = E[0];
        U[JB][1] = E[1];
        if constexpr (NC > 1) {
            // W[r][2q+e] = U[2q+e][r], which lives in lane (2q+e, r/2), register r%2
            const int s0 = 8 * q + (r >> 1), s1 = s0 + 4;
            const double a0 = shfl(E[0], s0), b0 = shfl(E[1], s0);
            const double a1 = shfl(E[0], s1), b1 = shfl(E[1], s1);
            const double W0 = (r & 1) ? b0 : a0, W1 = (r & 1) ? b1 : a1;
#pragma unroll
            for (int i = 1; i < NC; ++i) {
                double c[2] = {0.0, 0.0};
                mma_nt(c, C[i][0], C[i][1], W0, W1);
                if constexpr (JB < Lean<NT>::NSM) {
                    *reinterpret_cast<double2*>(Lsm + Lean<NT>::sidx(JB + i, JB) * 64 + 2 * lane) = make_double2(c[0], c[1]);
                } else {
                    R[Lean<NT>::ridx(JB + i, JB)][0] = c[0];
                    R[Lean<NT>::ridx(JB + i, JB)][1] = c[1];
                }
            }
        }
        if constexpr (FWD) {
            double acc = 0.0;
#pragma unroll
            for (int J = 0; J < JB; ++J) {              // w_J = D^-1 z_J of the finished blocks comes back from shared memory
                const double2 t = lean_tile<NT>(Lsm, R, JB, J, lane);
                const double2 wJ = *reinterpret_cast<const double2*>(zscr + 8 * J + 2 * q);
                acc = fma(t.x, wJ.x, fma(t.y, wJ.y, acc));
            }
            double rr = rhs[8 * JB + r];
            if (JB > 0) rr -= quadreduce(acc);
            const double z0 = colreduce(U[JB][0] * rr), z1 = colreduce(U[JB][1] * rr);       // z = L^-1 rhs (unit L)
            const double2 dj = *reinterpret_cast<const double2*>(dinv + 8 * JB + 2 * q);
            if (r == 0) *reinterpret_cast<double2*>(zscr + 8 * JB + 2 * q) = make_double2(z0 * dj.x, z1 * dj.y);
            __syncwarp();
        }
        lean_steps<NT, JB + 1, FWD>(load, Lsm, R, U, ok, logdet, want_logdet, r, q, lane, rhs, zscr, dinv);
    }
}

// Backward substitution L^T x = z with the lean factor; z = L^{-1} rhs was parked in `zscr` (8 NT doubles of shared
// memory owned by this warp) by lean_steps<FWD>.  x is returned row-replicated: xr[I] = x[8 I + r] on every lane of row r.
template <int NT>
__device__ __forceinline__ void lean_solve(const double* __restrict__ Lsm, const double (&R)[Lean<NT>::RDIM][2],
                                           const double (&U)[NT][2], const double* __restrict__ dinv, double (&xr)[NT], int r,
                                           int q, int lane, const double* __restrict__ zscr) {
    __syncwarp();
#pragma unroll
    for (int jb = NT - 1; jb >= 0; --jb) {
        double c0 = 0.0, c1 = 0.0;
#pragma unroll
        for (int I = jb + 1; I < NT; ++I) {
            const double2 t = lean_tile<NT>(Lsm, R, I, jb, lane);
            c0 = fma(t.x, xr[I], c0);
            c1 = fma(t.y, xr[I], c1);
        }
        const double2 w = *reinterpret_cast<const double2*>(zscr + 8 * jb + 2 * q);      // D^-1 L^-1 rhs
        double z0 = w.x, z1 = w.y;
        if (jb < NT - 1) {
            const double2 dj = *reinterpret_cast<const double2*>(dinv + 8 * jb + 2 * q);
            z0 = fma(-dj.x, colreduce(c0), z0); z1 = fma(-dj.y, colreduce(c1), z1);
        }
        xr[jb] = quadreduce(fma(U[jb][0], z0, U[jb][1] * z1));
    }
    __syncwarp();
}

// ------------------------------------------------------------------------------------------
// Wide variants of the factorisation: the same left-looking blocked L D L^T, the same arithmetic per tile and per pivot as
// lean_steps / lean_solve, but every tile of the factor lives in this warp's slice Lw of the global workspace (NTRI
// tiles; a lane only ever reads back what it stored itself) and the block-column loops are run-time loops.  The
// diagonal slot of block JB holds U = L_d^{-T}.  x replaces w = D^-1 L^-1 rhs in `zscr`.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ double2 wtile(const double* Lw, int I, int J, int lane) {
    return *reinterpret_cast<const double2*>(Lw + (size_t)tri(I, J) * 64 + 2 * lane);
}
template <int NT, bool FWD, class Load>
__device__ __forceinline__ void wide_factor(Load& load, double* Lw, bool& ok, double& logdet, bool want_logdet, int r, int q,
                                            int lane, const double* rhs, double* zscr, double* dinv) {
    for (int JB = 0; JB < NT; ++JB) {
        const int NC = NT - JB;
        double C[NT][2];
#pragma unroll
        for (int i = 0; i < NT; ++i)
            if (i < NC) { const double2 t = load(JB + i, JB); C[i][0] = t.x; C[i][1] = t.y; }
        for (int K = 0; K < JB; ++K) {
            const double2 y = wtile(Lw, JB, K, lane);
            const double2 dk = *reinterpret_cast<const double2*>(dinv + 8 * K + 2 * q);
            const double ys0 = y.x * dk.x, ys1 = y.y * dk.y;
#pragma unroll
            for (int i = 0; i < NT; ++i)
                if (i < NC) {
                    const double2 x = i == 0 ? y : wtile(Lw, JB + i, K, lane);
                    mma_nt(C[i], -x.x, -x.y, ys0, ys1);
                }
        }
        double E[2];
        E[0] = (r == 2 * q) ? 1.0 : 0.0;
        E[1] = (r == 2 * q + 1) ? 1.0 : 0.0;
        double(&P0)[2] = C[0];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int jq = j >> 1, je = j & 1;
            const double ajj = shfl(P0[je], 4 * j + jq);
            const double lk0 = shfl(P0[je], 8 * q + jq);
            const double lk1 = shfl(P0[je], 8 * q + 4 + jq);
            const int src = (lane & ~3) | jq;
            const double lp = shfl(P0[je], src);
            const double le = shfl(E[je], src);
            if (!(ajj > 0.0)) ok = false;
            if (want_logdet) logdet += log(ajj);
            const double inv = rcp_nr(ajj);
            const double p0 = lp * lk0, p1 = lp * lk1, e0 = le * lk0, e1 = le * lk1;
            if (2 * q > j) { P0[0] = fma(-p0, inv, P0[0]); E[0] = fma(-e0, inv, E[0]); }
            if (2 * q + 1 > j) { P0[1] = fma(-p1, inv, P0[1]); E[1] = fma(-e1, inv, E[1]); }
            if (lane == 0) dinv[8 * JB + j] = inv;
        }
        __syncwarp();
        *reinterpret_cast<double2*>(Lw + (size_t)tri(JB, JB) * 64 + 2 * lane) = make_double2(E[0], E[1]);
        if (NC > 1) {
            const int s0 = 8 * q + (r >> 1), s1 = s0 + 4;
            const double a0 = shfl(E[0], s0), b0 = shfl(E[1], s0);
            const double a1 = shfl(E[0], s1), b1 = shfl(E[1], s1);
            const double W0 = (r & 1) ? b0 : a0, W1 = (r & 1) ? b1 : a1;
#pragma unroll
            for (int i = 1; i < NT; ++i)
                if (i < NC) {
                    double c[2] = {0.0, 0.0};
                    mma_nt(c, C[i][0], C[i][1], W0, W1);
                    *reinterpret_cast<double2*>(Lw + (size_t)tri(JB + i, JB) * 64 + 2 * lane) = make_double2(c[0], c[1]);
                }
        }
        if constexpr (FWD) {
            double acc = 0.0;
            for (int J = 0; J < JB; ++J) {
                const double2 t = wtile(Lw, JB, J, lane);
                const double2 wJ = *reinterpret_cast<const double2*>(zscr + 8 * J + 2 * q);
                acc = fma(t.x, wJ.x, fma(t.y, wJ.y, acc));
            }
            double rr = rhs[8 * JB + r];
            if (JB > 0) rr -= quadreduce(acc);
            const double z0 = colreduce(E[0] * rr), z1 = colreduce(E[1] * rr);
            const double2 dj = *reinterpret_cast<const double2*>(dinv + 8 * JB + 2 * q);
            if (r == 0) *reinterpret_cast<double2*>(zscr + 8 * JB + 2 * q) = make_double2(z0 * dj.x, z1 * dj.y);
            __syncwarp();
        }
    }
}

template <int NT>
__device__ __forceinline__ void wide_solve(const double* Lw, const double* dinv, double* zscr, int r, int q, int lane) {
    __syncwarp();
    for (int jb = NT - 1; jb >= 0; --jb) {
        double c0 = 0.0, c1 = 0.0;
        for (int I = jb + 1; I < NT; ++I) {
            const double2 t = wtile(Lw, I, jb, lane);
            const double xI = zscr[8 * I + r];
            c0 = fma(t.x, xI, c0);
            c1 = fma(t.y, xI, c1);
        }
        const double2 w = *reinterpret_cast<const double2*>(zscr + 8 * jb + 2 * q);
        double z0 = w.x, z1 = w.y;
        if (jb < NT - 1) {
            const double2 dj = *reinterpret_cast<const double2*>(dinv + 8 * jb + 2 * q);
            z0 = fma(-dj.x, colreduce(c0), z0); z1 = fma(-dj.y, colreduce(c1), z1);
        }
        const double2 U = wtile(Lw, jb, jb, lane);
        const double x = quadreduce(fma(U.x, z0, U.y * z1));
        __syncwarp();                                      // every lane holds w_jb before x_jb takes its place
        if (q == 0) zscr[8 * jb + r] = x;
        __syncwarp();
    }
}

// Wide H-pass: Z = V'^T diag(w) V' in blocks of 4 x 4 tiles per warp (accumulators in registers), every block a full
// pass over V' in k order -- one warp per tile, hence one fixed summation order and no reduction between warps.
template <int NT>
__device__ __forceinline__ void hpass_wide(const double* __restrict__ Vt, const double* __restrict__ wrow, int n_kt, double* Zf,
                                           int warp, int lane, int r, int q, int offY0, int offY1) {
    constexpr int BI = 4, BJ = 4;
    constexpr int NBI = (NT + BI - 1) / BI, NBJ = (NT + BJ - 1) / BJ;
    int cnt = 0;
    for (int bi = 0; bi < NBI; ++bi)
        for (int bj = 0; bj < NBJ && BJ * bj <= BI * bi + BI - 1; ++bj, ++cnt) {
            if (cnt % NWARP != warp) continue;
            const int I0 = bi * BI, J0 = bj * BJ;
            double z[BI][BJ][2];
#pragma unroll
            for (int i = 0; i < BI; ++i)
#pragma unroll
                for (int j = 0; j < BJ; ++j) { z[i][j][0] = 0.0; z[i][j][1] = 0.0; }
            // fragments of the block's rows (I0..) and columns (J0..) of one k-tile, both omega halves; the next k-tile is
            // fetched from L2 while the MMAs of the current one issue
            auto fetch = [&](int kt, double2& w, double (&fi)[2][BI], double (&fj)[2][BJ]) {
                if (kt >= n_kt) return;
                w = *reinterpret_cast<const double2*>(wrow + kt * 8 + 2 * q);
                const double* tile = Vt + (size_t)kt * NT * 64;
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int off = e ? offY1 : offY0;
#pragma unroll
                    for (int i = 0; i < BI; ++i) fi[e][i] = (I0 + i < NT) ? tile[(I0 + i) * 64 + off] : 0.0;
#pragma unroll
                    for (int j = 0; j < BJ; ++j) fj[e][j] = (J0 + j < NT) ? tile[(J0 + j) * 64 + off] : 0.0;
                }
            };
            double2 wn = make_double2(0.0, 0.0);
            double fin[2][BI], fjn[2][BJ];
            fetch(0, wn, fin, fjn);
            for (int kt = 0; kt < n_kt; ++kt) {
                const double2 w = wn;
                double fi[2][BI], fj[2][BJ];
#pragma unroll
                for (int e = 0; e < 2; ++e) {
#pragma unroll
                    for (int i = 0; i < BI; ++i) fi[e][i] = fin[e][i];
#pragma unroll
                    for (int j = 0; j < BJ; ++j) fj[e][j] = fjn[e][j];
                }
                fetch(kt + 1, wn, fin, fjn);
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const double we = e ? w.y : w.x;
#pragma unroll
                    for (int i = 0; i < BI; ++i)
#pragma unroll
                        for (int j = 0; j < BJ; ++j)
                            if (J0 + j <= I0 + i && I0 + i < NT) dmma(z[i][j], we * fi[e][i], fj[e][j]);
                }
            }
#pragma unroll
            for (int i = 0; i < BI; ++i)
#pragma unroll
                for (int j = 0; j < BJ; ++j) {
                    const int I = I0 + i, J = J0 + j;
                    if (J <= I && I < NT) {
                        *reinterpret_cast<double2*>(Zf + (size_t)(I * NT + J) * 64 + 2 * lane) = make_double2(z[i][j][0], z[i][j][1]);
                        if (I != J) {
                            Zf[(size_t)(J * NT + I) * 64 + (2 * q) * 8 + r] = z[i][j][0];
                            Zf[(size_t)(J * NT + I) * 64 + (2 * q + 1) * 8 + r] = z[i][j][1];
                        }
                    }
                }
        }
    __syncthreads();
}

// The pointwise map of the cost pass for this lane's two omega rows: H = D e^x (plus-minus: D (e^x - e^-x)), w = dH/dx,
// and the entropy terms added to sacc.
template <bool pm>
__device__ __forceinline__ void pointwise(double x0, double x1, double2 Dv, double (&Hv)[2], double (&Wv)[2], double& sacc) {
    // the two (plus-minus: four) exponentials of this lane as independent straight-line chains; the rare
    // huge arguments (overflowing pump trials) take the library path
    double ex2[2], em2[2] = {0.0, 0.0};
    if (__any_sync(0xffffffffu, mx::exp_is_special(x0) || mx::exp_is_special(x1))) {
        ex2[0] = exp(x0); ex2[1] = exp(x1);
        if (pm) { em2[0] = exp(-x0); em2[1] = exp(-x1); }
    } else {
        ex2[0] = mx::exp_main(x0); ex2[1] = mx::exp_main(x1);
        if (pm) { em2[0] = mx::exp_main(-x0); em2[1] = mx::exp_main(-x1); }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const double Dk = i ? Dv.y : Dv.x;
        const double x = i ? x1 : x0;
        const double ex = ex2[i];
        double H, W, st_;
        if (!pm) {
            // H = D e^x ; S += H - D - H log(H/D), safelog clamp at 1e-100  (functions.py:53-56,508-510)
            H = Dk * ex; W = H;
            const double lg = (ex <= 1e-100) ? -230.25850929940458 : x;
            st_ = H - Dk - H * lg;
        } else {
            // H = D (e^x - e^-x) ; w = D (e^x + e^-x) ; S = S_n(H+) + S_n(H-)   (functions.py:544-564,778-786)
            const double em = em2[i];
            const double Hp = Dk * ex, Hm = Dk * em;
            H = Hp - Hm; W = Hp + Hm;
            const double lp = (ex <= 1e-100) ? -230.25850929940458 : x;
            const double lm = (em <= 1e-100) ? -230.25850929940458 : -x;
            st_ = (Hp - Dk - Hp * lp) + (Hm - Dk - Hm * lm);
        }
        if (Dk == 0.0) { H = 0.0; W = 0.0; st_ = 0.0; }   // padded rows / missing tile
        sacc += st_;
        Hv[i] = H; Wv[i] = W;
    }
}

// ------------------------------------------------------------------------------------------
// H-pass tile ownership: rows of the lower triangle owned by tile-half 0 (the rest belongs to half 1)
// ------------------------------------------------------------------------------------------
__host__ __device__ constexpr unsigned rowmask0(int NT) {
    return NT == 4 ? 0x9u : NT == 5 ? 0x14u : NT == 6 ? 0x30u : NT == 7 ? 0x61u : NT == 8 ? 0xC4u : NT == 9 ? 0x190u :
           NT == 10 ? 0x380u : 0u;
}
template <int NT, int TH>
__host__ __device__ constexpr bool owns(int I) { return (((rowmask0(NT) >> I) & 1u) != 0u) == (TH == 0); }
template <int NT, int TH>
__host__ __device__ constexpr int maxrow() {
    int m = 0;
    for (int I = 0; I < NT; ++I) if (owns<NT, TH>(I)) m = I;
    return m;
}

template <int NT, int TH>
__device__ __forceinline__ void hpass_ktile(const double* __restrict__ tile0, double w0, double w1, int offY0, int offY1,
                                            double (&zacc)[Lay<NT>::NTRI][2]) {
    constexpr int MR = maxrow<NT, TH>();
#pragma unroll
    for (int e = 0; e < 2; ++e) {
        const int off = e ? offY1 : offY0;
        const double we = e ? w1 : w0;
        double fr[MR + 1];
#pragma unroll
        for (int jt = 0; jt <= MR; ++jt) fr[jt] = tile0[jt * 64 + off];
#pragma unroll
        for (int I = 0; I <= MR; ++I) {
            if (owns<NT, TH>(I)) {
                const double sc = we * fr[I];
#pragma unroll
                for (int J = 0; J <= I; ++J) dmma(zacc[tri(I, J)], sc, fr[J]);
            }
        }
    }
}


// ------------------------------------------------------------------------------------------
// V' streaming pipeline: 1-D TMA bulk copies into NSTAGE staging buffers, full/empty mbarriers.
// Chunks are numbered globally (g) across passes so that the mbarrier phases stay consistent.
// ------------------------------------------------------------------------------------------
template <int NT>
struct Pipe {
    static constexpr int NSTAGE = Lay<NT>::NST;
    double* stage0;
    uint64_t* full;
    uint64_t* empty;
    int tid, lane, n_kt, nch;

    // Vt = the V' buffer of the spectrum in work (whitening groups bring their own, MxProblem.vt_index)
    __device__ __forceinline__ void issue(int c, unsigned g, const double* __restrict__ Vt) const {      // thread 0 only
        const int st = g % NSTAGE;
        const int t0 = c * CH;
        const int nt = min(CH, n_kt - t0);
        const uint32_t bytes = (uint32_t)nt * NT * 64 * sizeof(double);
        mbar_expect_tx(full + st, bytes);
        bulk_g2s(stage0 + st * Lay<NT>::STAGE_D, Vt + (size_t)t0 * NT * 64, bytes, full + st);
    }
    // all threads; the staging area may have been used as scratch (generic proxy) since the last pass
    __device__ __forceinline__ void begin(unsigned g0, const double* __restrict__ Vt) const {
        __syncthreads();
        if (tid == 0) {
            fence_proxy_async();
            for (int c = 0; c < NSTAGE - 1 && c < nch; ++c) issue(c, g0 + c, Vt);
        }
    }
    // wait for chunk c of the pass; thread 0 first tops the pipeline up (the stage of chunk c-1 is refilled)
    __device__ __forceinline__ const double* wait(int c, unsigned g0, const double* __restrict__ Vt, long long* pf = nullptr) const {
        const unsigned g = g0 + c;
#ifdef MX_TPROF
        // diagnostics build: pf[0] time thread 0 waits for a free stage, pf[1] time it waits for data, pf[2] steps,
        // pf[4] / pf[5] issue -> completion latency of the copies it had to wait for (sum / count); pf[8..] issue stamps
        if (tid == 0 && pf) {
            const long long t0 = clock64();
            const int cn = c + NSTAGE - 1;
            if (cn < nch) {
                if (c >= 1) mbar_wait(empty + (g - 1) % NSTAGE, ((g - 1) / NSTAGE) & 1);
                pf[0] += clock64() - t0;
                issue(cn, g0 + cn, Vt);
                pf[8 + (g0 + cn) % NSTAGE] = clock64();
            }
            const long long w0 = clock64();
            mbar_wait(full + g % NSTAGE, (g / NSTAGE) & 1);
            const long long w1 = clock64();
            pf[1] += w1 - w0; pf[2] += 1;
            if (w1 - w0 > 60 && c >= NSTAGE - 1) { pf[4] += w1 - pf[8 + g % NSTAGE]; pf[5] += 1; }
        } else
#endif
        if (tid == 0) {
            const int cn = c + NSTAGE - 1;
            if (cn < nch) {
                if (c >= 1) mbar_wait(empty + (g - 1) % NSTAGE, ((g - 1) / NSTAGE) & 1);
                issue(cn, g0 + cn, Vt);
            }
        }
        __syncwarp();
        mbar_wait(full + g % NSTAGE, (g / NSTAGE) & 1);
        return stage0 + (g % NSTAGE) * Lay<NT>::STAGE_D;
    }
    __device__ __forceinline__ void release(int c, unsigned g0) const {
        const unsigned g = g0 + c;
        __syncwarp();
        if (lane == 0) mbar_arrive(empty + g % NSTAGE);
    }
};

// H-pass body for one tile half: Z_owned += sum_k w_k V'[k, I] V'[k, J] over this warp's k-tiles (two of every chunk:
// k-group kg takes tiles 2 kg and 2 kg + 1), then the k-groups are added in a fixed order into Zfull (all NT x NT
// tiles, C layout, symmetric fill).
template <int NT, int TH>
__device__ __forceinline__ void hpass_body(const Pipe<NT>& pipe, const double* __restrict__ Vt, unsigned g0, const double* __restrict__ wrow, int kg,
                                           int lane, int r, int q, int offY0, int offY1, double* __restrict__ Zf) {
    constexpr int NTRI = Lay<NT>::NTRI;
    const int n_kt = pipe.n_kt, nch = pipe.nch;
    double zacc[NTRI][2];
#pragma unroll
    for (int I = 0; I < NT; ++I)
        if (owns<NT, TH>(I)) {
#pragma unroll
            for (int J = 0; J <= I; ++J) { zacc[tri(I, J)][0] = 0.0; zacc[tri(I, J)][1] = 0.0; }
        }
    static_assert(CH == 2 * NKG, "two k-tiles of every chunk per k-group");
    // w of this lane's two omega rows (2q, 2q+1) of both tiles, prefetched one chunk ahead (the scratch rows live in
    // L2: the load must not sit between the arrival of a chunk and its first MMA)
    auto loadw = [&](int kt) -> double2 {
        if (kt < n_kt) return *reinterpret_cast<const double2*>(wrow + kt * 8 + 2 * q);
        return make_double2(0.0, 0.0);
    };
    double2 wa = loadw(2 * kg), wb = loadw(2 * kg + 1);
    for (int c = 0; c < nch; ++c) {
        const double* stage = pipe.wait(c, g0, Vt);
        const int kt = c * CH + 2 * kg;
        const double2 na = loadw(kt + CH), nb = loadw(kt + CH + 1);
        if (kt < n_kt) hpass_ktile<NT, TH>(stage + (2 * kg) * NT * 64, wa.x, wa.y, offY0, offY1, zacc);
        if (kt + 1 < n_kt) hpass_ktile<NT, TH>(stage + (2 * kg + 1) * NT * 64, wb.x, wb.y, offY0, offY1, zacc);
        wa = na; wb = nb;
        pipe.release(c, g0);
    }
    // The k-groups are added in the fixed order ((g0 + g1) + g2) + ... (deterministic sums).  Groups 1.. park their
    // partial tiles behind Zfull -- the staging ring, J and the trial vectors are all dead during an H-pass and
    // contiguous -- and the two warps of group 0 finish the sum, write Zfull and mirror it.
    double* const slots = Zf + NT * NT * 64;
    __syncthreads();                                       // every warp is done with the staging area
    if (kg > 0) {
#pragma unroll
        for (int I = 0; I < NT; ++I)
            if (owns<NT, TH>(I)) {
#pragma unroll
                for (int J = 0; J <= I; ++J)
                    *reinterpret_cast<double2*>(slots + ((kg - 1) * NTRI + tri(I, J)) * 64 + 2 * lane) =
                        make_double2(zacc[tri(I, J)][0], zacc[tri(I, J)][1]);
            }
    }
    __syncthreads();
    if (kg == 0) {
#pragma unroll
        for (int I = 0; I < NT; ++I)
            if (owns<NT, TH>(I)) {
#pragma unroll
                for (int J = 0; J <= I; ++J) {
                    double2 vv = make_double2(zacc[tri(I, J)][0], zacc[tri(I, J)][1]);
#pragma unroll
                    for (int g = 0; g < NKG - 1; ++g) {
                        const double2 o = *reinterpret_cast<const double2*>(slots + (g * NTRI + tri(I, J)) * 64 + 2 * lane);
                        vv.x += o.x; vv.y += o.y;
                    }
                    *reinterpret_cast<double2*>(Zf + (I * NT + J) * 64 + 2 * lane) = vv;
                    if (I != J) {                          // mirror: tile (J, I) = transpose
                        Zf[(J * NT + I) * 64 + (2 * q) * 8 + r] = vv.x;
                        Zf[(J * NT + I) * 64 + (2 * q + 1) * 8 + r] = vv.y;
                    }
                }
            }
    }
    __syncthreads();
}

// ------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------
// CTAs per SM the instantiation is compiled for: the target (CTAS_PER_SM), or what its shared memory allows
template <int NT>
__host__ __device__ constexpr int ctas_per_sm() {
    if (is_wide(NT)) return 1;                // the block accumulators of the wide H-pass need the full register file
    int n = (228 * 1024) / (Lay<NT>::total * (int)sizeof(double) + 1024);
    if (n > CTAS_PER_SM) n = CTAS_PER_SM;
    return n < 1 ? 1 : n;
}

// VAR = cost-function variant (MX_VARIANT_*), MARQ = Marquardt damping: compile-time, so that the code of the other
// variants (the second pair of exponentials and the H rows of plus-minus, Bryan's scaling) costs the default path neither
// registers nor instructions
template <int NT, int VAR, bool MARQ>
__global__ void __launch_bounds__(NTHR, ctas_per_sm<NT>()) sweep2_kernel(const SweepArgs a) {
    using LY = Lay<NT>;
    using LN = Lean<NT>;
    constexpr int SP = LY::SP;
    constexpr int NTRI = LY::NTRI;
    extern __shared__ __align__(128) double sm[];
    Ctl& ctl = *reinterpret_cast<Ctl*>(sm + LY::o_ctl);
    uint64_t* bar_full = reinterpret_cast<uint64_t*>(sm + LY::o_bar);
    uint64_t* bar_empty = bar_full + LY::NST;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int r = lane >> 2, q = lane & 3;
    const int s = a.n_sv;
    const double eps_nu = a.nu * 2.220446049250313e-16;
    constexpr bool pm = VAR == MX_VARIANT_PLUSMINUS;
    constexpr bool bryan = VAR == MX_VARIANT_BRYAN;
    const int n_kt = a.n_kt;
    const int nch = (n_kt + CH - 1) / CH;
    const size_t rowlen = (size_t)n_kt * 8;
    double* const wscr = a.scratch + (size_t)blockIdx.x * (pm ? 2 : 1) * NROWS * rowlen;   // [NROWS][rowlen] (+ H rows for plusminus)
    double* const hscr = wscr + (size_t)NROWS * rowlen;

    constexpr bool WIDE = LY::WIDE;
    // wide instantiations: Zfull, J and one factor per warp in this CTA's slice of the global workspace
    double* const wZ = WIDE ? a.wide + (size_t)blockIdx.x * (size_t)a.wide_stride : nullptr;
    double* const wJ = wZ + NT * NT * 64;
    double* const wL = wJ + (size_t)(1 + warp) * NTRI * 64;
    auto Zfull = [&]() -> double* { if constexpr (WIDE) return wZ; else return sm + LY::o_stage; };
    auto Jtiles = [&]() -> double* { if constexpr (WIDE) return wJ; else return sm + LY::o_J; };

    const int offX = tile_off(r, 2 * q);
    const int offY0 = tile_off(2 * q + 0, r);
    const int offY1 = tile_off(2 * q + 1, r);

    if (tid == 0) {
        for (int i = 0; i < LY::NST; ++i) { mbar_init(bar_full + i, 1); mbar_init(bar_empty + i, NWARP); }
        ctl.gchunk = 0;
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    for (int i = tid; i < SP; i += NTHR) {
        const double x = (i < s && !a.per_spec_xi) ? a.xi[i] : 0.0;
        sm[LY::o_xi + i] = x;
        sm[LY::o_lam + i] = x * x;
    }
    __syncthreads();

    const Pipe<NT> pipe{sm + LY::o_stage, bar_full, bar_empty, tid, lane, n_kt, nch};
    const double* Vsp = a.Vt;                  // V' of the spectrum in work
    const double* Dsp = a.D;
    // phase timers: thread 0 charges the cycles since the previous tick to phase k (only when the caller asked
    // for them: MxSweepOut.phase_cycles)
    const bool timing = a.o_phase != nullptr;
    auto tick = [&](int k) {
#ifndef MX_TPROF
        if (timing && tid == 0) { const long long t = clock64(); ctl.tph[k] += t - ctl.t_last; ctl.t_last = t; }
#else
        (void)k;
#endif
    };
    const uint64_t keep_pol = l2_evict_last_policy();

    // ---- T-pass: evaluate the cost function at the trial vectors tb[0..7] ---------------------------
    // Per unique trial u < nuniq: yb[u], uchi2, uS, uQ, and w (and H) rows in scratch.
    // Warp w works on k-tile (NWARP c + w) of chunk c: x = V' t for the eight trials (M of the MMA), the pointwise map
    // H = D e^x with its entropy terms, y += H^T V'.
    auto tpass = [&]() {
        const unsigned g0 = ctl.gchunk;
        const int nuniq = ctl.nuniq;
        double yacc[NT][2];
#pragma unroll
        for (int jt = 0; jt < NT; ++jt) { yacc[jt][0] = 0.0; yacc[jt][1] = 0.0; }
        double sacc = 0.0;
        const bool live = r < nuniq;
        double* const wrow = wscr + (size_t)(live ? ctl.urow[r] : 0) * rowlen;
        double* const hrow = hscr + (size_t)(live ? ctl.urow[r] : 0) * rowlen;
        // D of this lane's two omega rows, fetched one step ahead (it may come from L2)
        auto loadD = [&](int kt) -> double2 {
            const int k0 = kt * 8 + 2 * q;
            double2 Dv = make_double2(0.0, 0.0);
            if (kt < n_kt) {
                if (k0 + 1 < a.n_omega) Dv = *reinterpret_cast<const double2*>(Dsp + k0);
                else if (k0 < a.n_omega) Dv.x = Dsp[k0];
            }
            return Dv;
        };
        if constexpr (WIDE) {
            __syncthreads();
            for (int kt = warp; kt < n_kt; kt += NWARP) {          // V' straight from L2, the trial vectors from shared memory
                const double* tile = Vsp + (size_t)kt * NT * 64;
                const double2 Dv = loadD(kt);
                double C0[2] = {0.0, 0.0}, C1[2] = {0.0, 0.0};
#pragma unroll
                for (int jt = 0; jt < NT; ++jt) {
                    const double2 tv = *reinterpret_cast<const double2*>(sm + LY::o_tb + r * SP + 8 * jt + 2 * q);
                    const double2 vv = *reinterpret_cast<const double2*>(tile + jt * 64 + offX);
                    dmma(C0, tv.x, vv.x);
                    dmma(C1, tv.y, vv.y);
                }
                double Hv[2], Wv[2];
                const int k0 = kt * 8 + 2 * q;
                pointwise<pm>(C0[0] + C1[0], C0[1] + C1[1], Dv, Hv, Wv, sacc);
                if (live) {
                    st_keep_v2(wrow + k0, Wv[0], Wv[1], keep_pol);
                    if (pm) st_keep_v2(hrow + k0, Hv[0], Hv[1], keep_pol);
                }
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int off = e ? offY1 : offY0;
#pragma unroll
                    for (int jt = 0; jt < NT; ++jt) dmma(yacc[jt], Hv[e], tile[jt * 64 + off]);
                }
            }
        } else {
        pipe.begin(g0, Vsp);
        double tA[NT][2];
#pragma unroll
        for (int jt = 0; jt < NT; ++jt) {
            const double2 tv = *reinterpret_cast<const double2*>(sm + LY::o_tb + r * SP + 8 * jt + 2 * q);
            tA[jt][0] = tv.x; tA[jt][1] = tv.y;
        }
        double2 Dv = loadD(warp);
        for (int c = 0; c < nch; ++c) {
#ifdef MX_TPROF
            const double* tile = pipe.wait(c, g0, Vsp, timing ? ctl.pf : nullptr) + warp * NT * 64;
#else
            const double* tile = pipe.wait(c, g0, Vsp) + warp * NT * 64;
#endif
            const int kt = c * CH + warp;
            const bool valid = kt < n_kt;
            const double2 Dn = loadD(kt + CH);
            double C0[2] = {0.0, 0.0}, C1[2] = {0.0, 0.0};
#pragma unroll
            for (int jt = 0; jt < NT; ++jt) {
                const double2 vv = *reinterpret_cast<const double2*>(tile + jt * 64 + offX);
                dmma(C0, tA[jt][0], vv.x);
                dmma(C1, tA[jt][1], vv.y);
            }
            double Hv[2], Wv[2];
            const int k0 = kt * 8 + 2 * q;
            pointwise<pm>(C0[0] + C1[0], C0[1] + C1[1], Dv, Hv, Wv, sacc);
            if (live && valid) {
                st_keep_v2(wrow + k0, Wv[0], Wv[1], keep_pol);
                if (pm) st_keep_v2(hrow + k0, Hv[0], Hv[1], keep_pol);
            }
            if (valid) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int off = e ? offY1 : offY0;
#pragma unroll
                    for (int jt = 0; jt < NT; ++jt) dmma(yacc[jt], Hv[e], tile[jt * 64 + off]);
                }
            }
            Dv = Dn;
            pipe.release(c, g0);
        }
        }
        __syncthreads();                                   // staging area is free: reuse as yred[NWARP][8][SP]
        if (tid == 0) ctl.gchunk = g0 + nch;
        double* yred = sm + LY::o_stage;
#pragma unroll
        for (int jt = 0; jt < NT; ++jt)
            *reinterpret_cast<double2*>(yred + (warp * 8 + r) * SP + 8 * jt + 2 * q) = make_double2(yacc[jt][0], yacc[jt][1]);
        {
            const double sq = quadreduce(sacc);
            if (q == 0) sm[LY::o_sred + warp * 8 + r] = sq;
        }
        __syncthreads();
        for (int i = tid; i < MAXB * SP; i += NTHR) {      // fixed-order tree over the warps (deterministic sums)
            const int b = i / SP, j = i - b * SP;
            const double* y0 = yred + b * SP + j;
            sm[LY::o_yb + i] = ((y0[0 * 8 * SP] + y0[1 * 8 * SP]) + (y0[2 * 8 * SP] + y0[3 * 8 * SP]))
                             + ((y0[4 * 8 * SP] + y0[5 * 8 * SP]) + (y0[6 * 8 * SP] + y0[7 * 8 * SP]));
        }
        __syncthreads();
        for (int u = warp; u < nuniq; u += NWARP) {        // chi2 = |Xi y - g~|^2 + c0  (functions.py:358-360 in singular space)
            double c2 = 0.0;
            for (int i = lane; i < s; i += 32) {
                const double rr = sm[LY::o_xi + i] * sm[LY::o_yb + u * SP + i] - sm[LY::o_gt + i];
                c2 = fma(rr, rr, c2);
            }
            c2 = warp_sum(c2) + ctl.c0;
            const double* sr = sm + LY::o_sred + u;
            const double S = ((sr[0] + sr[8]) + (sr[16] + sr[24])) + ((sr[32] + sr[40]) + (sr[48] + sr[56]));
            if (lane == 0) {
                ctl.uchi2[u] = c2; ctl.uS[u] = S;
                ctl.uQ[u] = ctl.ufail[u] ? nan("") : 0.5 * c2 * a.eta - ctl.alpha * S;   // maxent_cost_function.py:82
            }
        }
        __syncthreads();
    };

    // ---- H-pass: Z = V'^T diag(w) V' with w from scratch row `row` -> Zfull (all NT x NT tiles, C layout) ----
    auto hpass = [&](int row) {
        const double* wrow = wscr + (size_t)row * rowlen;
        if constexpr (WIDE) {
            __syncthreads();
            hpass_wide<NT>(Vsp, wrow, n_kt, wZ, warp, lane, r, q, offY0, offY1);
        } else {
            const unsigned g0 = ctl.gchunk;
            pipe.begin(g0, Vsp);
            const int kg = warp >> 1, th = warp & 1;
            double* Zf = sm + LY::o_stage;
            if (th == 0) hpass_body<NT, 0>(pipe, Vsp, g0, wrow, kg, lane, r, q, offY0, offY1, Zf);
            else hpass_body<NT, 1>(pipe, Vsp, g0, wrow, kg, lane, r, q, offY0, offY1, Zf);
            if (tid == 0) ctl.gchunk = g0 + nch;
            __syncthreads();
        }
    };

    // ---- gradient: u = eta Xi (Xi y - g~) + alpha v ; f = Z u (or u for Bryan) ; maxf -------------------
    auto gradient = [&]() {
        const double alpha = ctl.alpha;
        for (int i = tid; i < SP; i += NTHR) {
            const double xi = sm[LY::o_xi + i];
            const double rr = xi * sm[LY::o_ycur + i] - sm[LY::o_gt + i];
            const double u = (i < s) ? a.eta * xi * rr + alpha * sm[LY::o_v + i] : 0.0;
            sm[LY::o_u + i] = u;
            if (bryan) {
                // f = g + alpha v ; the reference solves the non-symmetric (eta Lambda Z + mu) dv = f
                // (bryan_cost_function.py:114-128).  With Lambda = Xi^2 the matrix is similar to the symmetric, well
                // scaled M = eta Xi Z Xi:  (M + mu) w = f / xi ,  dv = xi w  -- same eigenvalues, uniform shift
                sm[LY::o_f + i] = u;
                sm[LY::o_rhs + i] = (i < s) ? u / xi : 0.0;
            }
        }
        __syncthreads();
        if (!bryan) {
            const double* Zf = Zfull();
            for (int I = warp; I < NT; I += NWARP) {
                double cf[2] = {0.0, 0.0};
#pragma unroll
                for (int K = 0; K < NT; ++K) {
                    const double2 z = *reinterpret_cast<const double2*>(Zf + (I * NT + K) * 64 + 2 * lane);
                    const double2 ub = *reinterpret_cast<const double2*>(sm + LY::o_u + 8 * K + 2 * q);
                    mma_nt(cf, z.x, z.y, ub.x, ub.y);
                }
                if (q == 0) { sm[LY::o_f + 8 * I + r] = cf[0]; sm[LY::o_rhs + 8 * I + r] = cf[0]; }
            }
            __syncthreads();
        }
        if (warp == 0) {
            double mf = 0.0;
            for (int i = lane; i < s; i += 32) mf = fmax(mf, fabs(sm[LY::o_f + i]));
            mf = warp_max(mf);
            if (lane == 0) ctl.maxf = mf;
        }
        __syncthreads();
    };

    // ---- J = eta Z Lambda Z + alpha Z (lower tiles, C layout) and its diagonal ---------------------------
    auto form_J = [&]() {
        const double* Zf = Zfull();
        const double alpha = ctl.alpha;
        // every warp owns the tiles t = warp, warp + NWARP, ...; G of them are formed at a time so that their accumulation
        // chains (NT dependent MMA pairs each) interleave
        constexpr int TPW = (NTRI + NWARP - 1) / NWARP;
        constexpr int G = WIDE ? 2 : (TPW < 4 ? TPW : 4);
        for (int t0 = warp; t0 < NTRI; t0 += NWARP * G) {
            int tI[G], tJ[G];
            double c[G][2];
            double2 zij[G];
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const int t = t0 + g * NWARP < NTRI ? t0 + g * NWARP : t0;     // a missing tile repeats the first one (not stored)
                int I = 0;
                while (tri(I + 1, 0) <= t) ++I;
                tI[g] = I; tJ[g] = t - tri(I, 0);
                c[g][0] = 0.0; c[g][1] = 0.0;
                zij[g] = *reinterpret_cast<const double2*>(Zf + (tI[g] * NT + tJ[g]) * 64 + 2 * lane);
            }
            if (!bryan) {
#pragma unroll
                for (int K = 0; K < NT; ++K) {
                    const double2 lm = *reinterpret_cast<const double2*>(sm + LY::o_lam + 8 * K + 2 * q);
#pragma unroll
                    for (int g = 0; g < G; ++g) {
                        const double2 zi = *reinterpret_cast<const double2*>(Zf + (tI[g] * NT + K) * 64 + 2 * lane);
                        const double2 zj = *reinterpret_cast<const double2*>(Zf + (tJ[g] * NT + K) * 64 + 2 * lane);
                        mma_nt(c[g], zi.x * lm.x, zi.y * lm.y, zj.x, zj.y);
                    }
                }
            }
#pragma unroll
            for (int g = 0; g < G; ++g) {
                const int t = t0 + g * NWARP;
                if (t >= NTRI) continue;
                const int I = tI[g], J = tJ[g];
                if (!bryan) {
                    c[g][0] = fma(a.eta, c[g][0], alpha * zij[g].x);       // maxent_cost_function.py:161-162 in singular space
                    c[g][1] = fma(a.eta, c[g][1], alpha * zij[g].y);
                } else {                                           // M = eta Xi Z Xi
                    const double xr_ = a.eta * sm[LY::o_xi + 8 * I + r];
                    const double2 xc = *reinterpret_cast<const double2*>(sm + LY::o_xi + 8 * J + 2 * q);
                    c[g][0] = xr_ * zij[g].x * xc.x; c[g][1] = xr_ * zij[g].y * xc.y;
                }
                if (I == J) {                                      // padded rows/columns: identity
                    const int i0 = 8 * I + r;
                    if (i0 >= s) { c[g][0] = (r == 2 * q) ? 1.0 : 0.0; c[g][1] = (r == 2 * q + 1) ? 1.0 : 0.0; }
                    else { if (8 * J + 2 * q >= s) c[g][0] = 0.0; if (8 * J + 2 * q + 1 >= s) c[g][1] = 0.0; }
                    if (r == 2 * q) sm[LY::o_jd + i0] = c[g][0];
                    if (r == 2 * q + 1) sm[LY::o_jd + i0] = c[g][1];
                } else {
                    if (8 * I + r >= s || 8 * J + 2 * q >= s) c[g][0] = 0.0;
                    if (8 * I + r >= s || 8 * J + 2 * q + 1 >= s) c[g][1] = 0.0;
                }
                *reinterpret_cast<double2*>(Jtiles() + (size_t)t * 64 + 2 * lane) = make_double2(c[g][0], c[g][1]);
            }
        }
        __syncthreads();
        if (warp == 0) {
            // floor for the planner's equivalence pre-test: two dampings can only give the same shifted diagonal
            // if they differ by less than ~2 ulps of min_k |J_kk| / (d shift_k / d mu) + mu, where the shift of entry k
            // is mu (all three cost functions; Bryan works on the symmetrised matrix) or mu J_kk (Marquardt)
            double m = INFINITY;
            for (int k = lane; k < s; k += 32) {
                const double jd = fabs(sm[LY::o_jd + k]);
                m = fmin(m, MARQ ? 1.0 : jd);
            }
            m = -warp_max(-m);
            if (lane == 0) ctl.jdmin = m;
        }
        __syncthreads();
    };

    // damping of diagonal entry i: mu * 1, or -- Marquardt's variant, levenberg_minimizer.py:181-185 -- mu * diag(J):
    // J_ii + mu * J_ii (for Bryan diag(eta Lambda Z) = diag(eta Xi Z Xi), so the symmetrised system carries the same shift)
    constexpr bool marq = MARQ;
    auto shift_of = [&](int i, double mu) -> double {
        return marq ? mu * sm[LY::o_jd + i] : mu;
    };

    // ---- P3: factorise J + shift(mu_u) and solve for every unique trial (one solver warp per matrix) -------
    auto solve_trials = [&]() {
        const int nuniq = ctl.nuniq;
        // every solver warp factorises one shifted Hessian at a time; the strictly-lower tiles of the leading block
        // columns are parked in this warp's slice of the idle staging ring
        constexpr int NSOLVE = WIDE ? NWARP : solver_warps(NT);
        double* const Lsm = sm + LY::o_stage + LY::STAGE_AREA - (warp + 1) * LN::NSMT * 64;
        for (int u = warp; u < nuniq && warp < NSOLVE; u += NSOLVE) {
            const double mu = ctl.umu[u];
            auto load = [&](int I, int J) -> double2 {
                double2 v = *reinterpret_cast<const double2*>(Jtiles() + (size_t)tri(I, J) * 64 + 2 * lane);
                if (I == J) {
                    const int i0 = 8 * I + r;
                    if (i0 < s) {
                        const double sh = shift_of(i0, mu);
                        if (r == 2 * q) v.x += sh;
                        if (r == 2 * q + 1) v.y += sh;
                    }
                }
                return v;
            };
            bool ok = true;
            double ld = 0.0;
            double* const trow = sm + LY::o_tb + u * SP;          // scratch for the forward substitution, then t = v - dv
            double* const dinv = sm + LY::o_yb + u * SP;          // 1 / d of the L D L^T factorisation (yb is dead here)
            double xr[NT];
            if constexpr (WIDE) {
                wide_factor<NT, true>(load, wL, ok, ld, false, r, q, lane, sm + LY::o_rhs, trow, dinv);
                ok = __all_sync(0xffffffffu, ok);
                wide_solve<NT>(wL, dinv, trow, r, q, lane);
#pragma unroll
                for (int I = 0; I < NT; ++I) xr[I] = trow[8 * I + r];
                __syncwarp();
            } else {
                double R[LN::RDIM][2];
                double U[NT][2];
                lean_steps<NT, 0, true>(load, Lsm, R, U, ok, ld, false, r, q, lane, sm + LY::o_rhs, trow, dinv);
                ok = __all_sync(0xffffffffu, ok);
                lean_solve<NT>(Lsm, R, U, dinv, xr, r, q, lane, trow);
            }
            if (q == 0) {
#pragma unroll
                for (int I = 0; I < NT; ++I) {
                    const int i0 = 8 * I + r;
                    const double dv = bryan ? sm[LY::o_xi + i0] * xr[I] : xr[I];
                    trow[i0] = ok ? sm[LY::o_v + i0] - dv : 0.0;
                }
            }
            if (lane == 0) ctl.ufail[u] = ok ? 0 : 1;
        }
        __syncthreads();
    };

    // ---- log det(I + eta Xi Z Xi / alpha) by warp 0 (probabilities.py:76-85 via Sylvester) -----------------
    auto logdet_prob = [&]() -> double {       // warp 0 only; returns NaN on a failed factorisation
        const double* Zf = Zfull();
        auto entry = [&](int I, int J) -> double2 {
            const double2 z = *reinterpret_cast<const double2*>(Zf + (I * NT + J) * 64 + 2 * lane);
            const int i0 = 8 * I + r, j0 = 8 * J + 2 * q;
            const double xi_i = sm[LY::o_xi + i0];
            double m0 = a.eta * xi_i * z.x * sm[LY::o_xi + j0] / ctl.alpha;
            double m1 = a.eta * xi_i * z.y * sm[LY::o_xi + j0 + 1] / ctl.alpha;
            if (i0 >= s || j0 >= s) m0 = 0.0;
            if (i0 >= s || j0 + 1 >= s) m1 = 0.0;
            if (i0 == j0) m0 += 1.0;
            if (i0 == j0 + 1) m1 += 1.0;
            return make_double2(m0, m1);
        };
        bool ok = true;
        double ld = 0.0;
        if constexpr (WIDE) {                              // J of the finished iteration is dead: park the tiles there
            wide_factor<NT, false>(entry, wJ, ok, ld, true, r, q, lane, nullptr, nullptr, sm + LY::o_yb);
        } else {
            double U[NT][2];
            double* const Lsm = sm + LY::o_J;
            double R[LN::RDIM][2];
            lean_steps<NT, 0, false>(entry, Lsm, R, U, ok, ld, true, r, q, lane, nullptr, nullptr, sm + LY::o_yb);
        }
        ok = __all_sync(0xffffffffu, ok);
        return ok ? ld : nan("");
    };

    // ==========================================================================================
    // main loop over spectra
    // ==========================================================================================
    for (;;) {
        __syncthreads();
        if (tid == 0) ctl.spec = atomicAdd(a.counter, 1);
        __syncthreads();
        const int sp = ctl.spec;
        if (sp >= a.B) break;
        Dsp = a.D + (a.per_spec ? (size_t)sp * ((a.n_omega + 1) & ~1) : 0);       // per-spectrum default model (Poorman off-diagonals)
        if (a.vt_index) Vsp = a.Vt + (size_t)a.vt_index[sp] * (size_t)a.vt_stride;   // the V' of this spectrum's whitening group
        const double* const v0sp = a.v0 + (a.per_spec ? (size_t)sp * s : 0);
        for (int i = tid; i < SP; i += NTHR) {
            const double v0 = i < s ? v0sp[i] : 0.0;
            sm[LY::o_v + i] = v0;
            sm[LY::o_gt + i] = i < s ? a.gt[(size_t)sp * s + i] : 0.0;
            if (a.per_spec_xi) {             // per-spectrum error scale: Xi_b = S / sigma_b (python/tau_maxent.py:227-251 per data set)
                const double x = i < s ? a.xi[(size_t)sp * s + i] : 0.0;
                sm[LY::o_xi + i] = x;
                sm[LY::o_lam + i] = x * x;
            }
        }
        for (int i = tid; i < MAXB * SP; i += NTHR) {
            const int b = i / SP, j = i - b * SP;
            sm[LY::o_tb + i] = (b == 0 && j < s) ? v0sp[j] : 0.0;
        }
        if (tid == 0) {
            ctl.ia = 0; ctl.it = 0; ctl.nq = 0; ctl.ns = 0; ctl.dir_up = 1; ctl.last_len = 99; ctl.ntrial = 1; ctl.nbatch = 1;
            ctl.alpha = a.alpha[a.per_spec_alpha ? (size_t)sp * a.n_alpha : 0]; ctl.c0 = a.c0[sp];
            ctl.lm.mu = a.mu0; ctl.lm.Q0 = nan(""); ctl.lm.phase = PH_FIRST;
            ctl.nuniq = 1; ctl.nb = 0; ctl.urow[0] = 0; ctl.ufail[0] = 0;
        }
        __syncthreads();
        // first evaluation at v0 (the reference's func_val = function(v), levenberg_minimizer.py:150)
        if (timing && tid == 0) { ctl.t_last = clock64(); for (int k = 0; k < 8; ++k) ctl.tph[k] = 0; }
#ifdef MX_TPROF
        if (timing && tid == 0) for (int k = 0; k < 16; ++k) ctl.pf[k] = 0;
#endif
        tpass();
        tick(PHT_TPASS);
        for (int i = tid; i < SP; i += NTHR) sm[LY::o_ycur + i] = sm[LY::o_yb + i];
        if (tid == 0) { ctl.chi2_cur = ctl.uchi2[0]; ctl.S_cur = ctl.uS[0]; ctl.cur_row = ctl.urow[0]; ctl.nq = 1; }
        __syncthreads();

        bool spectrum_done = false;
        while (!spectrum_done) {
            tick(PHT_OTHER);
            hpass(ctl.cur_row);
            tick(PHT_HPASS);
            // ---- convergence test / alpha loop (levenberg_minimizer.py:157-174, maxent_loop.py:241-266) ----
            for (;;) {
                gradient();
                tick(PHT_GRAD);
                if (tid == 0) {
                    LM& L = ctl.lm;
                    L.Q1 = 0.5 * ctl.chi2_cur * a.eta - ctl.alpha * ctl.S_cur;
                    // MaxDerivative(1e-4) | RelativeFunctionChange(1e-16)   (levenberg_minimizer.py:103-106)
                    //   | FunctionChange(x) when asked for (convergence_methods.py:100-110)
                    const bool conv = (ctl.maxf < a.conv_maxd) || (fabs(fabs(L.Q0 - L.Q1) / L.Q1) < a.conv_relq) ||
                                      (fabs(L.Q0 - L.Q1) < a.conv_absq);
                    ctl.conv = conv ? 1 : 0;
                    ctl.action = ((conv && ctl.it >= a.miniter) || ctl.it >= a.maxiter) ? 1 : 0;
                }
                __syncthreads();
                if (!ctl.action) break;
                // ---- this alpha is finished: probability, outputs ----
                const size_t o = (size_t)sp * a.n_alpha + ctl.ia;
                if (a.want_prob) {
                    if (warp == 0) {
                        const double ld = logdet_prob();
                        if (lane == 0) ctl.pq[0] = ld;
                    }
                    __syncthreads();
                }
                if (tid == 0) {
                    const double logp = a.want_prob ? -0.5 * ctl.pq[0] - ctl.lm.Q1 - log(ctl.alpha) : nan("");
                    const bool hit_max = ctl.it >= a.maxiter;
                    a.o_chi2[o] = ctl.chi2_cur;
                    a.o_S[o] = ctl.S_cur;
                    a.o_Q[o] = ctl.lm.Q1;
                    if (a.o_logp) a.o_logp[o] = logp;
                    if (a.o_niter) a.o_niter[o] = hit_max ? a.maxiter : ctl.it + 1;
                    if (a.o_nq) a.o_nq[o] = ctl.nq;
                    if (a.o_ns) a.o_ns[o] = ctl.ns;
                    if (a.o_ntrial) a.o_ntrial[o] = ctl.ntrial;
                    if (a.o_nbatch) a.o_nbatch[o] = ctl.nbatch;
                    if (a.o_status) a.o_status[o] = (!hit_max && ctl.conv) ? MX_STATUS_CONVERGED : 0;
                }
                if (a.o_v) for (int i = tid; i < s; i += NTHR) __stcs(a.o_v + o * s + i, sm[LY::o_v + i]);
                if (a.o_A) {                                   // A = H / delta  (functions.py:947-952)
                    const double* hr = (pm ? hscr : wscr) + (size_t)ctl.cur_row * rowlen;
                    for (int k = tid; k < a.n_omega; k += NTHR) __stcs(a.o_A + o * a.n_omega + k, hr[k] / a.delta[k]);
                }
                __syncthreads();
                if (tid == 0) {
                    ctl.ia++;
                    if (ctl.ia < a.n_alpha) {
                        ctl.alpha = a.alpha[(a.per_spec_alpha ? (size_t)sp * a.n_alpha : 0) + ctl.ia];
                        ctl.lm.mu = a.mu0; ctl.lm.Q0 = nan(""); ctl.it = 0; ctl.nq = 1; ctl.ns = 0; ctl.dir_up = 1; ctl.last_len = 99;
                        ctl.ntrial = 0; ctl.nbatch = 0;
                    }
                }
                __syncthreads();
                if (ctl.ia >= a.n_alpha) {
                    if (timing && tid == 0) {
                        tick(PHT_OTHER);
#ifdef MX_TPROF
                        for (int k = 0; k < 8; ++k) a.o_phase[(size_t)sp * 8 + k] = ctl.pf[k];
#else
                        for (int k = 0; k < 8; ++k) a.o_phase[(size_t)sp * 8 + k] = ctl.tph[k];
#endif
                    }
                    spectrum_done = true;
                    break;
                }
            }
            if (spectrum_done) break;
            tick(PHT_OTHER);
            form_J();
            tick(PHT_FORMJ);
            // ---- one Levenberg iteration: speculative batches until the damping search is decided ----
            if (tid == 0) { ctl.lm.Q0 = ctl.lm.Q1; ctl.lm.phase = PH_FIRST; ctl.nb = 0; ctl.nuniq = 0; ctl.urow[ID_CARRY] = -1; ctl.ns_it0 = ctl.ns; }
            __syncthreads();
            for (;;) {
                if (warp == 0)
                    replay_and_plan<MARQ>(ctl, a, eps_nu, s, SP, lane, sm + LY::o_jd, sm + LY::o_tb, sm + LY::o_yb, sm + LY::o_ctb,
                                          sm + LY::o_cy, timing, tick);
                __syncthreads();
                tick(PHT_PLAN);
                if (ctl.conv) break;
                for (int i = tid; i < MAXB * SP; i += NTHR) if (i >= ctl.nuniq * SP) sm[LY::o_tb + i] = 0.0;
                solve_trials();
                tick(PHT_SOLVE);
                {
                    // every factorisation of the batch failed (J + mu not positive definite numerically, the early
                    // part of a pump): all Q are NaN by definition, no pass over V' is needed
                    bool allfail = true;
                    for (int u = 0; u < ctl.nuniq; ++u) allfail = allfail && (ctl.ufail[u] != 0);
                    if (allfail) {
                        if (tid < ctl.nuniq) { ctl.uQ[tid] = nan(""); ctl.uchi2[tid] = nan(""); ctl.uS[tid] = nan(""); }
                        __syncthreads();
                    } else {
                        tpass();
                    }
                    tick(PHT_TPASS);
                }
            }
            // ---- accept: v -= dv ; the accepted trial becomes the current point (levenberg_minimizer.py:239-243) ----
            {
                const int id = ctl.lm.dv;
                // the accepted trial vector t = v - dv IS the new v (same subtraction, same operands); a failed solve has
                // dv = 0 by definition
                const double* tt = (id == ID_CARRY) ? sm + LY::o_ctb : sm + LY::o_tb + id * SP;
                const double* yy = (id == ID_CARRY) ? sm + LY::o_cy : sm + LY::o_yb + id * SP;
                const bool moved = ctl.ufail[id] == 0;
                for (int i = tid; i < SP; i += NTHR) {
                    if (i < s && moved) sm[LY::o_v + i] = tt[i];
                    sm[LY::o_ycur + i] = yy[i];
                }
                __syncthreads();
                if (tid == 0) {
                    ctl.chi2_cur = ctl.uchi2[id]; ctl.S_cur = ctl.uS[id]; ctl.cur_row = ctl.urow[id];
                    ctl.it++;
                    ctl.nq++;                                    // the reference re-evaluates func_val = function(v)
                    ctl.dir_up = (ctl.lm.nuf == a.nu) ? 1 : 0;
                    ctl.last_len = ctl.ns - ctl.ns_it0;
                }
                __syncthreads();
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// host-side launch
// ------------------------------------------------------------------------------------------
template <int NT, int VAR, bool MARQ>
int launch_variant(const SweepArgs& a, cudaStream_t stream, bool query, size_t bytes, int sms, int* o_grid) {
    auto kernel = sweep2_kernel<NT, VAR, MARQ>;
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) {
        if (query) { cudaGetLastError(); if (o_grid) *o_grid = 0; return MX_OK; }
        return MX_ERR_CUDA;
    }
    // persistent CTAs: as many as are resident at once (registers and shared memory decide; ctas_per_sm<NT>() is what
    // the instantiation was compiled for)
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, NTHR, bytes) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        per_sm = 1;
    }
    if (const char* e = getenv("MX_MAX_CTAS_PER_SM")) {        // diagnostics: uncontended phase times
        const int cap = atoi(e);
        if (cap >= 1 && cap < per_sm) per_sm = cap;
    }
    int grid = per_sm * sms;
    if (grid > a.B) grid = a.B;
    if (grid < 1) grid = 1;
    if (o_grid) *o_grid = grid;
    if (query) return MX_OK;
    kernel<<<grid, NTHR, bytes, stream>>>(a);
    return cudaGetLastError() == cudaSuccess ? MX_OK : MX_ERR_CUDA;
}

template <int NT>
int launch_sweep2(const SweepArgs& a, cudaStream_t stream, bool query, int* o_smem, int* o_grid) {
    const size_t bytes = (size_t)Lay<NT>::total * sizeof(double);
    if (o_smem) *o_smem = (int)bytes;
    if (query && !o_grid) return MX_OK;                        // pure introspection: no device needed
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { if (query) { *o_grid = 0; return MX_OK; } return MX_ERR_NO_DEVICE; }
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (a.marquardt) {
        switch (a.variant) {
            case MX_VARIANT_NORMAL: return launch_variant<NT, MX_VARIANT_NORMAL, true>(a, stream, query, bytes, sms, o_grid);
            case MX_VARIANT_PLUSMINUS: return launch_variant<NT, MX_VARIANT_PLUSMINUS, true>(a, stream, query, bytes, sms, o_grid);
            default: return launch_variant<NT, MX_VARIANT_BRYAN, true>(a, stream, query, bytes, sms, o_grid);
        }
    }
    switch (a.variant) {
        case MX_VARIANT_NORMAL: return launch_variant<NT, MX_VARIANT_NORMAL, false>(a, stream, query, bytes, sms, o_grid);
        case MX_VARIANT_PLUSMINUS: return launch_variant<NT, MX_VARIANT_PLUSMINUS, false>(a, stream, query, bytes, sms, o_grid);
        default: return launch_variant<NT, MX_VARIANT_BRYAN, false>(a, stream, query, bytes, sms, o_grid);
    }
}

constexpr int threads_per_cta() { return NTHR; }

}  // namespace mx2
