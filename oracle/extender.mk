# TEST INFRASTRUCTURE ONLY, for cudaextender (make -f extender.mk [oracle_ext] [ref_ext]):
#   liboracle_extender.so   - the CPU restatement of the ungapped X-drop extender (extender_oracle.cpp)
#   _ref/libgwref_ext.so     - the UNMODIFIED reference cudaextender, compiled for sm_100a from the sources where they lie under
#                              $(REF) (no copies) with the flags of Makefile's libgwref.so, + the ref_extender_capi.cu driver;
#                              skipped when the sources are absent (a prebuilt file travels)
include Makefile
.DEFAULT_GOAL := all_ext

EXT_INC  := $(INC) -I $(REF)/cudaextender/include
EXT_OBJS := $(OBJ)/cudaextender/src/ungapped_xdrop.cu.o $(OBJ)/cudaextender/src/ungapped_xdrop_kernels.cu.o \
            $(OBJ)/ext/extender.o $(OBJ)/ext/cudaextender.o $(OBJ)/ext/cudautils.o $(OBJ)/ext/logging.o $(OBJ)/ext/ref_extender_capi.o

.PHONY: all_ext oracle_ext ref_ext
all_ext: oracle_ext ref_ext
oracle_ext: liboracle_extender.so

liboracle_extender.so: extender_oracle.cpp
	$(CXX) -O2 -std=c++17 -fPIC -shared -ffp-contract=off -o $@ $^

ifneq ($(wildcard $(REF)/cudaextender/src/ungapped_xdrop.cu),)
ref_ext: $(OUT)/libgwref_ext.so
else
ref_ext:
	@echo "reference sources absent - using prebuilt $(OUT)/libgwref_ext.so if present"
endif

$(OBJ)/cudaextender/src/%.cu.o: $(REF)/cudaextender/src/%.cu
	@mkdir -p $(dir $@)
	$(NVCC) $(NVFLAGS) $(EXT_INC) -c $< -o $@

$(OBJ)/ext/%.o: $(REF)/cudaextender/src/%.cpp
	@mkdir -p $(dir $@)
	$(NVCC) -x cu $(NVFLAGS) -include stdexcept $(EXT_INC) -c $< -o $@

$(OBJ)/ext/%.o: $(REF)/common/base/src/%.cpp
	@mkdir -p $(dir $@)
	$(NVCC) -x cu $(NVFLAGS) $(EXT_INC) -c $< -o $@

$(OBJ)/ext/ref_extender_capi.o: ref_extender_capi.cu
	@mkdir -p $(dir $@)
	$(NVCC) $(NVFLAGS) $(EXT_INC) -c $< -o $@

$(OUT)/libgwref_ext.so: $(EXT_OBJS)
	$(NVCC) -shared -gencode arch=compute_100a,code=sm_100a -o $@ $^ -lcudart
