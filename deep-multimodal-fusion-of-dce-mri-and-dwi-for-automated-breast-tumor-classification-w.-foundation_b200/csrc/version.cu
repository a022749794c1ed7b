#include "b200_fusion.h"
extern "C" int b200_abi_version(void) { return 25; }
