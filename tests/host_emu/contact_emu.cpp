// TEST-ONLY host emulation of the contact plant: compiles the product header wbc_quadruped_dob_b200/csrc/wbc_contact.cuh
// (contact_step_instance and its Goldfarb-Idnani contact QP) with g++, so that the kernel's arithmetic and decisions can be checked
// against an independent reference on a machine without a GPU.  It is NOT linked into libwbc_b200.so; GPU tests call the CUDA
// kernel through the C ABI instead.
#include "../../wbc_quadruped_dob_b200/csrc/wbc_contact.cuh"

extern "C" {

// n instances, all arrays SoA [k][ld]; the state advances in place.  Optional arrays may be NULL, as in wbc_plant_contact_step.
void emu_contact_step(const wbc::Params* P, const wbc::ContactParams* cp, int n, long ld, double* base_pos, double* base_rot, double* base_rpy,
                      double* base_vel, double* q, double* dq, double* foot_force, const double* tau, const double* push, const double* ground_z,
                      const double* mu, int* contact, double* diag, int* status, int nsub)
{
    wbc::ContactIO io;
    io.base_pos = base_pos; io.base_rot = base_rot; io.base_rpy = base_rpy; io.base_vel = base_vel; io.q = q; io.dq = dq;
    io.foot_force = foot_force; io.tau = tau; io.push = push; io.ground_z = ground_z; io.mu = mu;
    io.contact = contact; io.diag = diag; io.status = status; io.ld = ld;
    for (long i = 0; i < n; i++) wbc::contact_step_instance(*P, *cp, io, i, nsub);
}

// One contact QP (contact_qp): H [nv*12] stride 12 (overwritten), g [nv], mu [nf]; warm [1] in/out; x [nv]; out [2]: iterations,
// KKT residual.  Returns the status.
int emu_contact_qp(double* H, const double* g, int nf, const double* mu, unsigned* warm, int max_iter, double* x, double* out)
{
    const wbc::ContactQpResult r = wbc::contact_qp(H, g, nf, mu, *warm, max_iter, x);
    out[0] = r.iters; out[1] = r.kkt;
    return r.status;
}

}
