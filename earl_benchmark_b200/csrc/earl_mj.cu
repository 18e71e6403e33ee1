// earl_mj.cu -- the exported entry points of include/earl_mj_b200.h: the Sawyer engine's primary capacity set (16 contacts,
// 64 rows, 16 environments in flight per SM), which runs both sawyer_door and sawyer_peg.  The env steps that outgrow it are
// re-stepped by the extra-large set's redo pass (earl_mj_xl.cu), so the small set is the faster choice for the peg as well
// (65,536 envs, steady window: 2.51e6 env-steps/s against 2.24e6 on the former 24-contact / 96-row set).
#include "earl_mj_impl.inc"
