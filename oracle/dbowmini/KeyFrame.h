// TEST INFRASTRUCTURE ONLY (oracle/).  The adapter build takes the KeyFrame stand-in from oracle/dbowshim/pre.hpp (force-included).
#pragma once
