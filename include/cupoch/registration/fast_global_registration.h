// Path-compatible with the reference header cupoch/registration/fast_global_registration.h; the declarations live in the single facade header.
#pragma once
#include "cupoch/cupoch_b200_facade.h"
