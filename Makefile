# Build of libcuadmm_b200.so + cuadmm_exe for sm_100a only (no other arch, no fallback).
NVCC      ?= /usr/local/cuda/bin/nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := -O3 -std=c++17 -lineinfo $(ARCH) -Xcompiler -fPIC,-O3,-Wall,-Wno-unused-function -Xptxas -v
SRC       := cuadmm_b200/csrc
LIBDIR    := cuadmm_b200/lib
OBJDIR    := build/obj
LIB       := $(LIBDIR)/libcuadmm_b200.so
EXE       := $(LIBDIR)/cuadmm_exe

CU_SRCS   := $(wildcard $(SRC)/*.cu)
CPP_SRCS  := $(filter-out $(SRC)/main.cpp,$(wildcard $(SRC)/*.cpp))
OBJS      := $(patsubst $(SRC)/%.cu,$(OBJDIR)/%.cu.o,$(CU_SRCS)) $(patsubst $(SRC)/%.cpp,$(OBJDIR)/%.cpp.o,$(CPP_SRCS))
HDRS      := $(wildcard $(SRC)/*.h) $(wildcard $(SRC)/*.cuh) include/cuadmm_b200.h

all: $(LIB) $(EXE)

$(OBJDIR)/%.cu.o: $(SRC)/%.cu $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> $(OBJDIR)/$*.ptxas.log || (cat $(OBJDIR)/$*.ptxas.log; false)

$(OBJDIR)/%.cpp.o: $(SRC)/%.cpp $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -x cu -c $< -o $@ 2> $(OBJDIR)/$*.cpp.log || (cat $(OBJDIR)/$*.cpp.log; false)

$(LIB): $(OBJS)
	@mkdir -p $(LIBDIR)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -lcudart $(EXTRA_LIBS)

$(EXE): $(SRC)/main.cpp $(LIB) $(HDRS)
	$(NVCC) -O2 -std=c++17 $(ARCH) -o $@ $(SRC)/main.cpp -L$(LIBDIR) -lcuadmm_b200 -Xlinker -rpath -Xlinker '$$ORIGIN'

clean:
	rm -rf build $(LIB) $(EXE)
.PHONY: all clean
