# oracle/strlist.mk — TEST INFRASTRUCTURE ONLY: the glue module that lets the compiled reference's AggList_string_int64 be driven from
# numpy (ref_strlist_shim.cpp).  Reuses the variables and rules of oracle/Makefile.
#
# usage:  make -C oracle -f strlist.mk ref    (everything `make -C oracle ref` builds, plus _ref/strlist_shim)

include Makefile

ref: _ref/strlist_shim$(EXT)

_ref/strlist_shim$(EXT): ref_strlist_shim.cpp _ref/obj/utl_string_utils.o $(REF)/src/superstring.hpp
	$(CXX) $(REF_CXXFLAGS) -I$(REF)/src -shared -o $@ ref_strlist_shim.cpp _ref/obj/utl_string_utils.o
