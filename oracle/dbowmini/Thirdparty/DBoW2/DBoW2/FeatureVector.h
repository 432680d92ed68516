// TEST INFRASTRUCTURE ONLY (oracle/).  Stand-in for DBoW2's FeatureVector: node id -> feature indices in insertion order.
#pragma once
#include <map>
#include <vector>

#include "BowVector.h"

namespace DBoW2 {

class FeatureVector : public std::map<NodeId, std::vector<unsigned int> > {
public:
    void addFeature(NodeId id, unsigned int i_feature) { (*this)[id].push_back(i_feature); }
};

}  // namespace DBoW2
