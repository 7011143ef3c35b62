# Included by build_ref_runtime.sh through CMAKE_PROJECT_PARSEC_INCLUDE.  The reference's CMakeLists.txt sets the
# install RPATH of libparsec to the absolute install prefix and adds every link directory to it, so the installed
# library would look for libparsec_b200.so in the checkout it was built in.  The install under oracle/_ref is built on
# one machine and run from another checkout on another, so at the end of configuration the RUNPATH of libparsec is made
# relative to the library itself: its own directory, then <repo>/parsec_b200, then the CUDA runtime.
function(pb2_relocatable_rpath)
  set_target_properties(parsec PROPERTIES
    INSTALL_RPATH "\$ORIGIN;\$ORIGIN/../../../../parsec_b200;${CUDAToolkit_LIBRARY_DIR}"
    INSTALL_RPATH_USE_LINK_PATH OFF)
endfunction()
cmake_language(DEFER DIRECTORY ${CMAKE_SOURCE_DIR} CALL pb2_relocatable_rpath)
