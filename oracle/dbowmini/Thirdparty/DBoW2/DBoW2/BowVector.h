// TEST INFRASTRUCTURE ONLY (oracle/).  Stand-in for DBoW2's BowVector with the types and the one member the adapter builds
// (oracle/Makefile target `adapt`) use, so that the product's drop-in sources compile and run without the reference tree.
#pragma once
#include <map>

namespace DBoW2 {

typedef unsigned int WordId;
typedef double WordValue;
typedef unsigned int NodeId;

class BowVector : public std::map<WordId, WordValue> {
public:
    void addWeight(WordId id, WordValue v) { (*this)[id] += v; }
};

}  // namespace DBoW2
