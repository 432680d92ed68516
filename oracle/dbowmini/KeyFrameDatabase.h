// TEST INFRASTRUCTURE ONLY (oracle/).  The KeyFrameDatabase class declaration with the reference's public interface and member
// names (include/KeyFrameDatabase.h), which integration/KeyFrameDatabase_borb.cc defines; used by the adapter build (oracle/Makefile
// target `adapt`) where the reference tree is absent.  KeyFrame / Frame come from oracle/dbowshim/pre.hpp.
#pragma once
#include <list>
#include <mutex>
#include <vector>

#include "ORBVocabulary.h"

namespace ORB_SLAM2 {

class KeyFrame;
class Frame;

class KeyFrameDatabase {
public:
    KeyFrameDatabase(const ORBVocabulary& voc);
    void add(KeyFrame* pKF);
    void erase(KeyFrame* pKF);
    void clear();
    std::vector<KeyFrame*> DetectLoopCandidates(KeyFrame* pKF, float minScore);
    std::vector<KeyFrame*> DetectRelocalizationCandidates(Frame* F);

protected:
    const ORBVocabulary* mpVoc;
    std::vector<std::list<KeyFrame*> > mvInvertedFile;
    std::mutex mMutex;
};

}  // namespace ORB_SLAM2
