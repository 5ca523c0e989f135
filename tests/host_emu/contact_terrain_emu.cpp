// TEST-ONLY host emulation of the contact plant's terrain form: compiles contact_step_instance<true> from the product header
// wbc_quadruped_dob_b200/csrc/wbc_contact.cuh with g++, so that the terrain kernel's arithmetic and decisions can be checked on a
// machine without a GPU.  It is NOT linked into libwbc_b200.so; GPU tests call the CUDA kernel through the C ABI instead.
#include "../../wbc_quadruped_dob_b200/csrc/wbc_contact.cuh"

extern "C" {

// n instances, all arrays SoA [k][ld]; the state advances in place.  terrain [40][ld] is required, plane_d [4][ld] may be NULL, as in
// wbc_plant_contact_step_terrain.
void emu_contact_terrain_step(const wbc::Params* P, const wbc::ContactParams* cp, int n, long ld, double* base_pos, double* base_rot,
                              double* base_rpy, double* base_vel, double* q, double* dq, double* foot_force, const double* tau,
                              const double* push, const double* terrain, const double* plane_d, int* contact, double* diag, int* status,
                              int nsub)
{
    wbc::ContactIO io;
    io.base_pos = base_pos; io.base_rot = base_rot; io.base_rpy = base_rpy; io.base_vel = base_vel; io.q = q; io.dq = dq;
    io.foot_force = foot_force; io.tau = tau; io.push = push; io.ground_z = plane_d; io.mu = nullptr;
    io.contact = contact; io.diag = diag; io.status = status; io.ld = ld;
    for (long i = 0; i < n; i++) wbc::contact_step_instance<true>(*P, *cp, io, i, nsub, terrain);
}

}
