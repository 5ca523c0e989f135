// TEST-ONLY host emulation of the gait generator: compiles gait_init_instance / gait_step_instance from the product header
// wbc_quadruped_dob_b200/csrc/wbc_gait.cuh with g++, so that the kernel's arithmetic and decisions can be checked against an
// independent reference on a machine without a GPU.  It is NOT linked into libwbc_b200.so; GPU tests call the CUDA kernels through
// the C ABI instead.
#include "../../wbc_quadruped_dob_b200/csrc/wbc_gait.cuh"

extern "C" {

// n robots, all arrays SoA [k][ld]; optional pointers may be NULL, as in wbc_gait_init / wbc_gait_step.
void emu_gait_init(const wbc::GaitParams* G, double dt, const wbc::GaitIO* io, int n)
{
    for (long i = 0; i < n; i++) wbc::gait_init_instance(*G, dt, *io, i);
}

void emu_gait_step(const wbc::GaitParams* G, double dt, const wbc::GaitIO* io, int n)
{
    for (long i = 0; i < n; i++) wbc::gait_step_instance(*G, dt, *io, i);
}

}
