// Internal declarations shared by the C-ABI translation units. Not installed.
#pragma once
#include <string>

#include "../../include/mfa_b200.h"
#include "kernels/attention_params.h"

namespace mfa {

extern thread_local std::string g_last_error;
int fail(int status, const std::string &message);

int memory_precision(const mfa_attention_descriptor_t &d, int operand);
int register_precision(const mfa_attention_descriptor_t &d, int operand);
int register_precision_for(const mfa_attention_descriptor_t &d, int operand, int type);
int select_backend(const mfa_attention_descriptor_t &d, int type);
const char *parameter_file(const mfa_attention_descriptor_t &d, int type);
unsigned parameter_table_generation();  // bumped by mfa_set_parameter_table: cached kernels of older tables are stale
int kernel_descriptor(const mfa_attention_descriptor_t &d, int type, mfa_attention_kernel_descriptor_t &out);
// MFA_SUCCESS when the current device is an sm_100 GPU, MFA_ERROR_NO_DEVICE (with the message set) otherwise
int check_device();

// Largest head dimension the compiled tcgen05 kernels cover (tcgen05_*.cu).
uint32_t tcgen05_forward_max_head();
uint32_t tcgen05_backward_max_head();

}  // namespace mfa
