# oracle/scale.mk — the body-scale (useScale) builds of the test infrastructure, next to oracle/Makefile:
#   make -C oracle -f scale.mk          the CPU oracle's scaled mode: _build/libsvsdf_scale_oracle{,_glibc}.so
#   make -C oracle -f scale.mk ref      + the reference's own source with `useScale` on: _ref/libref_path_scaled_{glibc,portable}.so
#                                       (only where /root/reference exists; outputs only under _ref/, git-ignored)
include Makefile

SCALE_OUT := _build/libsvsdf_scale_oracle.so _build/libsvsdf_scale_oracle_glibc.so
scale: $(SCALE_OUT)
.DEFAULT_GOAL := scale
_build/libsvsdf_scale_oracle.so: scale_oracle.cpp $(HDRS)
	mkdir -p _build
	$(CXX) $(CXXFLAGS) -shared -o $@ scale_oracle.cpp
_build/libsvsdf_scale_oracle_glibc.so: scale_oracle.cpp $(HDRS)
	mkdir -p _build
	$(CXX) $(CXXFLAGS) -DORACLE_GLIBC_SINCOS -shared -o $@ scale_oracle.cpp

# The reference's path with `#define useScale true` and getScale from a spec.  ref_path_shim.cpp is compiled from a copy under
# _ref/scaled/, so that its two quoted includes that change resolve next to it: _ref/gen/sw_macros.inc (ref_scale/sw_macros.inc:
# the verbatim macros, then useScale redefined true) and _ref/gen/sw_methods.inc (ref_scale/sw_methods.inc: getScale from the
# spec, then the verbatim methods without the cut getScale block, _ref/gen/sw_methods_scaled.inc by ref_scale_extract.py).
# -DNDEBUG (REF_PATH_FLAGS) matters here: the scaled getStateOnTrajStamp overloads assert the inverted condition.
_ref/gen/sw_methods_scaled.inc: _ref/gen/.stamp ref_scale_extract.py
	python3 ref_scale_extract.py --gen _ref/gen
_ref/scaled/ref_path_shim.cpp: ref_path_shim.cpp ref_scale/sw_macros.inc ref_scale/sw_methods.inc
	mkdir -p _ref/scaled/_ref/gen
	cp ref_path_shim.cpp $@
	cp ref_scale/sw_macros.inc ref_scale/sw_methods.inc _ref/scaled/_ref/gen/
REF_SCALED_DEPS := $(REF_PATH_DEPS) ref_path_scaled.cpp _ref/scaled/ref_path_shim.cpp _ref/gen/sw_methods_scaled.inc
_ref/libref_path_scaled_glibc.so: $(REF_SCALED_DEPS)
	$(CXX) $(REF_PATH_FLAGS) -shared -o $@ ref_path_scaled.cpp
_ref/libref_path_scaled_portable.so: $(REF_SCALED_DEPS)
	$(CXX) $(REF_PATH_FLAGS) -mfma -DREF_LIBM_PORTABLE -shared -o $@ ref_path_scaled.cpp
ref_scaled: _ref/libref_path_scaled_glibc.so _ref/libref_path_scaled_portable.so
