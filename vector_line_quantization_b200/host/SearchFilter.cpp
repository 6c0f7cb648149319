#include "SearchFilter.h"

namespace faiss {
namespace gpu {

DeviceSelector checkSearchSelector(const IDSelector* sel) {
  DeviceSelector s;
  while (const IDSelectorNot* no = dynamic_cast<const IDSelectorNot*>(sel)) {  // Not(Not(x)) folds to x
    s.invert = !s.invert;
    sel = no->sel;
  }
  s.range = dynamic_cast<const IDSelectorRange*>(sel);
  s.batch = dynamic_cast<const IDSelectorBatch*>(sel);
  s.bitmap = dynamic_cast<const IDSelectorBitmap*>(sel);
  VLQ_THROW_IF_NOT_MSG(s.range || s.batch || s.bitmap,
                       "search: the selector must be an IDSelectorRange, IDSelectorBatch or IDSelectorBitmap, or an "
                       "IDSelectorNot of one of them");
  VLQ_THROW_IF_NOT_MSG(!s.bitmap || s.bitmap->n == 0 || s.bitmap->bitmap, "search: IDSelectorBitmap has a null bitmap");
  return s;
}

}  // namespace gpu
}  // namespace faiss
