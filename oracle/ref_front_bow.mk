# TEST INFRASTRUCTURE ONLY.  oracle/_ref/libref_front_bow.so: libref_front.so's recipe (Makefile) with ref_front_bow_wrap.cpp as
# the wrapper -- it includes ref_front_wrap.cpp and adds the reference's SearchByBoW, both overloads.  Only possible where
# $(REF) exists.  usage: make -C oracle -f ref_front_bow.mk REF=<reference root> _ref/libref_front_bow.so
include Makefile
_ref/libref_front_bow.so: ref_front_bow_wrap.cpp ref_front_wrap.cpp cvcompat/opencv2/opencv.hpp eigencompat/Eigen/Core eigencompat/sophus/se3.hpp liborb_oracle.so \
                          $(REF)/src/ORBmatcher.cc $(REF)/src/Frame.cc $(REF)/src/KeyFrame.cc $(REF)/src/MapPoint.cc $(REF)/src/ORBextractor.cc $(REF)/src/CameraModels/Pinhole.cpp
	mkdir -p _ref/front_bow
	for f in src/ORBmatcher.cc src/Frame.cc src/KeyFrame.cc src/MapPoint.cc src/ORBextractor.cc src/CameraModels/Pinhole.cpp \
	         Thirdparty/DBoW2/DBoW2/BowVector.cpp Thirdparty/DBoW2/DBoW2/FeatureVector.cpp; do \
	  $(CXX) $(EDGE_FLAGS) $(FRONT_INC) -c $(REF)/$$f -o _ref/front_bow/`basename $$f | sed 's/\..*//'`.o || exit 1; done
	$(CXX) $(EDGE_FLAGS) $(FRONT_INC) -c ref_front_bow_wrap.cpp -o _ref/front_bow/wrap.o
	$(CXX) -shared -Wl,-Bsymbolic -Wl,--exclude-libs,ALL -o _ref/front_bow/probe.so _ref/front_bow/*.o -L. -l:liborb_oracle.so
	( echo '#include <stdio.h>'; echo '#include <stdlib.h>'; \
	  echo 'static void off_path(const char* s) { fprintf(stderr, "libref_front_bow: %s is outside the compared path", s); fputc(10, stderr); abort(); }'; \
	  nm -D --undefined-only _ref/front_bow/probe.so | awk '{print $$2}' | grep -E '^_ZNK?(9ORB_SLAM3|5DBoW2)' | \
	  awk '{printf "void %s(void) { off_path(\"%s\"); }\n", $$1, $$1}' ) > _ref/front_bow/off_path.c
	rm -f _ref/front_bow/probe.so
	gcc -O1 -fPIC -c _ref/front_bow/off_path.c -o _ref/front_bow/off_path.o
	$(CXX) -shared -Wl,-Bsymbolic -Wl,--exclude-libs,ALL -o $@ _ref/front_bow/*.o -L. -l:liborb_oracle.so -Wl,-rpath,'$$ORIGIN/..'
	rm -rf _ref/front_bow
