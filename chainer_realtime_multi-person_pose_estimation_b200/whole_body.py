"""Face and hand keypoints of every person of a frame in two batches: the per-person loop of the reference's demo.py
(:30-57) with one FaceDetector.detect_batch and one HandDetector.detect_batch call in place of up to three detector
calls per person.

    person_pose_array, _ = pose_detector(img)
    people = detect_face_and_hands(img, person_pose_array, pose_detector, face_detector, hand_detector)
    # people[i] = {"face": (keypoints, bbox) or None, "left": (keypoints, bbox) or None, "right": ...}

The crops are the reference loop's: per person get_unit_length, crop_face, then crop_hands, in that order.  The order
matters because crop_hands moves the hand joint of `person_pose` (a view into person_pose_array) towards the elbow
direction in place (pose_detector.py:377-392), exactly as the reference loop leaves it."""


def detect_face_and_hands(img, person_pose_array, pose_detector, face_detector, hand_detector):
    people = []
    faces, face_owner = [], []
    hands, hand_types, hand_owner = [], [], []
    for p, person_pose in enumerate(person_pose_array):
        people.append({"face": None, "left": None, "right": None})
        unit_length = pose_detector.get_unit_length(person_pose)
        cropped_face_img, bbox = pose_detector.crop_face(img, person_pose, unit_length)
        if cropped_face_img is not None:
            faces.append(cropped_face_img)
            face_owner.append((p, bbox))
        crops = pose_detector.crop_hands(img, person_pose, unit_length)
        for side in ("left", "right"):
            if crops[side] is not None:
                hands.append(crops[side]["img"])
                hand_types.append(side)
                hand_owner.append((p, side, crops[side]["bbox"]))
    for keypoints, (p, bbox) in zip(face_detector.detect_batch(faces), face_owner):
        people[p]["face"] = (keypoints, bbox)
    for keypoints, (p, side, bbox) in zip(hand_detector.detect_batch(hands, hand_types), hand_owner):
        people[p][side] = (keypoints, bbox)
    return people
