// Capacity set "extra large" (56 contacts, 224 rows, 6 environments in flight per SM) of the Sawyer engine: only its redo
// pass is compiled with a host side (earl_mjx_redo_pass) -- mj_redo_kernel re-steps the environments whose substep
// overflowed the primary set (earl_mj.cu, earl_mj_impl.inc).
#define MJ_CAPSET_XL 1
#define mj mjx  // the engine namespace of this translation unit (earl::mjx): Model and Work differ from the primary set's
#include "earl_mj_impl.inc"
