# Builds the B200-native libmultiexp.so (sm_100a only) and the CPU-side oracles.
NVCC      ?= nvcc
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Xcompiler -Wall -Xcompiler -Wno-unknown-pragmas -diag-suppress 128
CSRC      := porla_b200/csrc
OBJDIR    := build
OBJS      := $(OBJDIR)/msm.o $(OBJDIR)/msm_bn254.o $(OBJDIR)/msm_secp.o $(OBJDIR)/abi.o $(OBJDIR)/multi.o $(OBJDIR)/abi_secp.o $(OBJDIR)/pint.o $(OBJDIR)/lat.o $(OBJDIR)/staging.o
HDRS      := $(wildcard $(CSRC)/*.cuh $(CSRC)/*.h $(CSRC)/*.hpp include/*.h)
LIB       := porla_b200/libmultiexp.so

REPLAY    := tools/replay_config1
REFHDR    := /root/reference/porla/Utils

all: $(LIB) oracle $(REPLAY)

# Config-1 replay harness (C++ caller of the C-ABI).  With the reference tree present the legacy prototypes come from
# the reference's own cgo header; otherwise from include/porla_multiexp.h (identical prototypes).
$(REPLAY): tools/replay_config1.cpp $(LIB) include/porla_multiexp.h
	@if [ -f $(REFHDR)/libmultiexp.h ]; then \
	  g++ -O2 -std=c++17 -DPORLA_USE_REFERENCE_HEADER -I$(REFHDR) -o $@ $< -Lporla_b200 -lmultiexp -Wl,-rpath,'$$ORIGIN/../porla_b200' -ldl -lpthread; \
	else \
	  g++ -O2 -std=c++17 -Iinclude -o $@ $< -Lporla_b200 -lmultiexp -Wl,-rpath,'$$ORIGIN/../porla_b200' -ldl -lpthread; \
	fi

$(OBJDIR)/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -c $< -o $@

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -lpthread

oracle:
	$(MAKE) -C oracle

clean:
	rm -rf $(OBJDIR) $(LIB) $(REPLAY)
	$(MAKE) -C oracle clean

.PHONY: all oracle clean
