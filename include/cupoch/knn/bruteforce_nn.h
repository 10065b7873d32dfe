// Path-compatible with the reference header cupoch/knn/bruteforce_nn.h; the declarations live in the single facade header.
#pragma once
#include "cupoch/cupoch_b200_facade.h"
